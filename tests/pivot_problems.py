"""Seeded problems whose Pade-13 denominators need row interchanges, and non-Hermitian Hamiltonians
(tests/test_gpu_pivoting.py, preconditions in tests/test_pivot_problems_cpu.py).

The random problems of tests/problems.py spread the norm of every operator over all entries; the denominator
Q = V - U of the Pade-13 approximant then stays diagonally dominant and partial pivoting never swaps a row.  The
families here concentrate the norm instead:

  H  Hermitian: a weak random drift (||dt H0||_1 = 0.3), real-control two-level couplings x (|a><b| + |b><a|) and one
     ladder drive a + a^dagger.  The first coupling follows deterministic plateaus that put the slices' ||A||_1 into all
     four LU brackets of the kernels: < 1.6 (no swap), [1.6, 2.5) (pivot-free LU where LAPACK swaps), [2.5, theta13)
     (pivoted LU, no squaring) and >= theta13 (squarings).
  N  non-Hermitian: real controls on a sub-diagonal shift and on one large off-diagonal entry, both without their
     adjoints.  Q is close to lower triangular with sub-diagonal entries larger than the diagonal: the row-major LU of
     the n <= 64 kernels swaps.  For n > 64 the entry sits above the diagonal instead, so that Q^T swaps too: cuBLAS
     getrf reads the row-major Q as column-major and factors Q^T.
  L  loss plus a non-adjoint complex drive pair: H = H0 - i Gamma / 2 + sum_k u_k C_k + conj(u_k) C'_k with
     C'_k = C_k^dagger + D_k.  The loss floor min(Gamma) / 2 exceeds the Hermitian part (i u D^dagger - i conj(u) D) / 2
     that the drives add to the generator, so state norms only decay.
  HS family H with plateau levels that keep every slice below ||A||_1 = 2.5, several in [1.6, 2.5) with row swaps:
     for n > 64 the plan then keeps its own block LU (pivoting inside the 64 x 64 diagonal blocks) instead of falling
     back to cuBLAS getrf / getrs, which a single slice at or above 2.5 triggers for the whole plan.
  E  classification edge: family H with an anti-Hermitian perturbation of one drift entry, relative size `edge` of
     the largest entry, on either side of the 1e-13 rule of `qocb_set_operators`.

Pure NumPy except the torch twins of the callables (imported lazily) and `magnus_matrices`, which uses the oracle."""
import math

import numpy as np

from tests.problems import haar_columns, one_norm, rand_herm

THETA13 = 5.371920351148152
NOPIV_NORM = 2.5            # QOCB_NOPIV_NORM (qoc_b200/csrc/expm_slice.cuh)
SWAP_FROM = 1.6             # a concentrated Hermitian coupling makes LAPACK swap from about here
BRACKETS = ("lt1.6", "nopiv", "pivoted", "scaled")

# plateau levels of the first H coupling: ||A||_1 of a plateau slice is about |level| + 0.3 (the drift) + the other drives
H_LEVELS = (0.8, 6.5, 1.75, -4.2, -2.05, -10.5, 2.9, 1.9, -3.6)
# HS: the same couplings, every slice below the pivot-free bound 2.5
HS_LEVELS = (0.8, 1.75, -1.9, 1.2, -1.7, 1.85)
# N: levels of the shift, held for two control points each and undone by the next level, so that the running sum of
# the shift amplitude (the shift commutes with itself) stays below ~3 and state norms stay bounded; levels of the single
# entry (nilpotent: exp(c E) = 1 + c E), which reach the squaring bracket
N_SHIFT_LEVELS = (0.7, -0.7, 2.4, -2.4, 3.1, -3.1, 1.9, -1.9, 2.8, -2.8)
N_ENTRY_LEVELS = (0.3, -0.3, 5.0, -5.0, -0.5, 0.5, 3.4, -3.4)
PLATEAU = 3
OWN_LU_BLOCK = 64           # n > 64: the large path; block size of its own LU


def bracket(norm):
    if norm < SWAP_FROM:
        return "lt1.6"
    if norm < NOPIV_NORM:
        return "nopiv"
    if norm < THETA13:
        return "pivoted"
    return "scaled"


def is_hermitian(h):
    """Python mirror of the classification in qocb_set_operators (qoc_b200/csrc/capi.cu)."""
    h = np.asarray(h, dtype=np.complex128)
    lo = np.tril_indices(h.shape[0])
    a, b = h[lo], h.T[lo]
    mx = max(np.max(np.abs(a.real) + np.abs(a.imag)), np.max(np.abs(b.real) + np.abs(b.imag)))
    dev = np.max(np.abs(a.real - b.real) + np.abs(a.imag + b.imag))
    return bool(dev <= 1e-13 * mx)


def coupling(n, a, b):
    m = np.zeros((n, n), dtype=np.complex128)
    m[a, b] = m[b, a] = 1.0
    return m


def ladder(n):
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(np.complex128)
    return a + a.T


def plateaus(levels, count, phase=0, length=PLATEAU):
    """`count` control values: each level held for `length` points, cycling (phase shifts the cycle)."""
    idx = (np.arange(count) // length + phase) % len(levels)
    return np.asarray(levels, dtype=np.float64)[idx]


class PivotProblem(object):
    """H = h0 + sum_k x_k ops[k] (real controls) or h0 + sum_k u_k ops[k] + conj(u_k) partners[k] (complex controls).
    The attribute names follow tests/problems.py:Problem (n, N, M, T, K, S, controls, initial_states, costs(mod), ...)."""

    def __init__(self, family, n, slices, K, S, order, F=0, seed=0, cost_eval_step=1, step_target=False, T=None,
                 edge=None):
        rng = np.random.default_rng(seed)
        self.family, self.n, self.N, self.K, self.S, self.order = family, n, slices + 1, K, S, order
        self.M = self.N
        self.T = float(slices) if T is None else float(T)
        dt = self.T / slices
        self.cost_eval_step, self.step_target, self.neglect_phase, self.F = cost_eval_step, step_target, False, F
        self.complex_controls = family == "L"
        h0 = rand_herm(rng, n)
        h0 = h0 * (0.3 / dt / one_norm(h0))
        self.partners = None
        t = np.arange(self.M)
        if family in ("H", "HS", "E"):
            ops = []
            pairs = [(0, 1 % n)] + [tuple(sorted(rng.choice(n, 2, replace=False))) if n > 1 else (0, 0) for _ in range(K)]
            for k in range(K):
                if k == K - 1 and K > 1:
                    ops.append(ladder(n) / one_norm(ladder(n)) if n > 1 else np.ones((1, 1), complex))
                else:
                    ops.append(coupling(n, *pairs[k]) if n > 1 else np.ones((1, 1), complex))
            ctl = np.zeros((self.M, K))
            ctl[:, 0] = plateaus(HS_LEVELS if family == "HS" else H_LEVELS, self.M)
            for k in range(1, K):
                ctl[:, k] = 0.25 * np.cos(0.37 * (k + 1) * t + k) / dt
            ctl[:, 0] /= dt
            if family == "E":
                i, j = (1, 0) if n > 1 else (0, 0)
                mx = np.max(np.abs(h0.real) + np.abs(h0.imag))
                eps = edge * mx / 2                        # the rule's deviation of the pair is 2 eps
                p = np.zeros((n, n), dtype=np.complex128)
                if i != j:
                    p[i, j], p[j, i] = eps, -eps
                else:
                    p[i, i] = 1j * eps
                h0 = h0 + p
        elif family == "N":
            h0 = h0 / 3                                     # ||dt H0||_1 = 0.1: conjugating it with the large shifts grows norms
            shift = np.diag(np.ones(n - 1), -1).astype(np.complex128) if n > 1 else np.ones((1, 1), complex)
            entry = np.zeros((n, n), dtype=np.complex128)
            row = min(n - 1, n // 2 + 1)
            if n <= OWN_LU_BLOCK:                           # below the diagonal: swaps in the row-major LU of Q
                entry[row, max(0, row - 2)] = 1.0
            else:                                           # above it: swaps in the LU of Q^T that getrf computes
                entry[max(0, row - 2), row] = 1.0
            ops = [shift, entry] + [rand_herm(rng, n) for _ in range(max(0, K - 2))]
            ops = [o if k < 2 else o * (0.1 / one_norm(o)) for k, o in enumerate(ops[:K])]
            ctl = np.zeros((self.M, K))
            ctl[:, 0] = plateaus(N_SHIFT_LEVELS, self.M, length=2) / dt
            if K > 1:
                ctl[:, 1] = plateaus(N_ENTRY_LEVELS, self.M, length=2) / dt
            for k in range(2, K):
                ctl[:, k] = np.cos(0.5 * t + k) / dt
        elif family == "L":
            gamma = np.linspace(1.0, 3.0, n) / self.T                 # sum over the pulse of dt * Gamma_ii = 1 ... 3
            h0 = h0 - 0.5j * np.diag(gamma)
            ops, partners = [], []
            for k in range(K):
                c = np.triu(rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n)), 1)
                c = c * (1.0 / dt / max(one_norm(c + c.conj().T), 1e-300))
                d = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
                # |u| <= 0.9 / dt below, so ||u D^dagger - conj(u) D||_2 <= 2 * 0.9 / dt * ||D||_2 = 0.2 * min(Gamma)
                d = d * (0.2 * gamma[0] * dt / 0.9 / 2 / np.linalg.norm(d, 2))
                ops.append(c)
                partners.append(c.conj().T + d)
            self.partners = np.array(partners).reshape(K, n, n)
            amp = 0.9 / dt * (0.4 + 0.6 * np.abs(np.sin(0.11 * t)))[:, None]
            ctl = amp * np.exp(1j * (0.3 * t[:, None] + np.arange(K)[None, :]))
        else:
            raise ValueError(family)
        self.h0 = h0
        self.ops = np.array(ops).reshape(K, n, n)
        self.controls = ctl
        self.initial_states = np.ascontiguousarray(haar_columns(rng, n, S).T)[:, :, None]
        self.target_states = np.ascontiguousarray(haar_columns(rng, n, S).T)[:, :, None]
        self.forbidden_states = None
        if F > 0:
            self.forbidden_states = np.array([np.ascontiguousarray(haar_columns(rng, n, min(F, n)).T)[:, :, None]
                                              for _ in range(S)])

    # -- callables -----------------------------------------------------------------------------------------------
    def hamiltonian_numpy(self):
        h0, ops, par = self.h0, self.ops, self.partners

        def hamiltonian(controls, time):
            h = h0
            if controls is None:
                return h
            for k in range(ops.shape[0]):
                h = h + controls[k] * ops[k]
                if par is not None:
                    h = h + np.conjugate(controls[k]) * par[k]
            return h
        return hamiltonian

    def hamiltonian_torch(self, h0=None):
        """the torch twin for the oracle; `h0` replaces the drift (ensemble members)."""
        import torch
        cdt = torch.complex128
        h0 = torch.as_tensor(self.h0 if h0 is None else h0, dtype=cdt)
        ops = torch.as_tensor(self.ops, dtype=cdt)
        par = None if self.partners is None else torch.as_tensor(self.partners, dtype=cdt)

        def hamiltonian(controls, time):
            h = h0
            if controls is None:
                return h
            for k in range(ops.shape[0]):
                h = h + controls[k] * ops[k]
                if par is not None:
                    h = h + torch.conj(controls[k]) * par[k]
            return h
        return hamiltonian

    def operators(self):
        """every matrix the plan classifies: the drift and the real-channel operators (complex controls: u = x + i y
        gives x (C + C') + y i (C - C'))."""
        if self.partners is None:
            return [self.h0] + list(self.ops)
        return [self.h0] + [c + p for c, p in zip(self.ops, self.partners)] + [1j * (c - p) for c, p in zip(self.ops, self.partners)]

    def costs(self, mod):
        out = []
        if self.step_target:
            out.append(mod.TargetStateInfidelityTime(self.N, self.target_states, cost_eval_step=self.cost_eval_step))
        else:
            out.append(mod.TargetStateInfidelity(self.target_states))
        if self.F > 0:
            out.append(mod.ForbidStates(self.forbidden_states, self.N, cost_eval_step=self.cost_eval_step, cost_multiplier=0.7))
        return out

    # -- the slices' Magnus matrices and their Pade denominators ------------------------------------------------------
    def magnus_matrices(self, order=None):
        """[N-1, n, n] Magnus matrices of the slices (oracle.magnus with the reference's control interpolation)."""
        import torch
        from oracle import qoc_oracle as orc
        order = self.order if order is None else order
        ham = self.hamiltonian_torch()
        xs = np.linspace(0, self.T, self.M)
        ctl = torch.as_tensor(self.controls)
        dt = self.T / (self.N - 1)
        out = []
        with torch.no_grad():
            for j in range(self.N - 1):
                gen = lambda t_: -1j * ham(orc.interpolate_linear_set(t_, xs, ctl), t_)
                out.append(orc.magnus(gen, dt, j * dt, order).numpy())
        return np.array(out)


def vanishing_pivot_theta():
    """the theta in (2.5, theta13) at which the Pade-13 denominator of A = -i theta (|0><1| + |1><0|) has a zero diagonal:
    with A^2 = -theta^2 on that pair, Q = c(theta) 1 + i theta d(theta) X, c(theta) = sum_k b_2k (-theta^2)^k.  Without a
    row exchange the elimination divides by c(theta) ~ 0."""
    from oracle.qoc_oracle import PADE13_B
    roots = np.roots([PADE13_B[2 * k] * (-1) ** k for k in range(6, -1, -1)])       # polynomial in theta^2
    th = sorted(math.sqrt(r.real) for r in roots if abs(r.imag) < 1e-9 and r.real > 0)
    return [t for t in th if NOPIV_NORM < t < THETA13][0]


def vanishing_pivot_matrix(n, eta=1e-10):
    """[n, n] generator whose Pade denominator needs a row exchange at the very first pivot (n >= 2).  The exact
    coupling alone is no test: its P and Q share the diagonal V, and elimination without exchange then cancels to the
    right answer.  A generic complex perturbation of relative size `eta` breaks that: without the exchange the solve
    loses ~1/eta * 1e-16 (tests/test_pivot_problems_cpu.py: test_vanishing_pivot_needs_exchange)."""
    rng = np.random.default_rng(100 + n)
    h = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    return -1j * vanishing_pivot_theta() * coupling(n, 0, 1) + h * (eta / one_norm(h))


def solve_without_exchange(q, p):
    """Q^-1 P by Gaussian elimination without row exchanges (what a kernel that skipped its pivot search computes)"""
    q, x = np.array(q, dtype=np.complex128), np.array(p, dtype=np.complex128)
    n = q.shape[0]
    for j in range(n):
        for i in range(j + 1, n):
            m = q[i, j] / q[j, j]
            q[i, j:] -= m * q[j, j:]
            x[i] -= m * x[j]
    for j in range(n - 1, -1, -1):
        x[j] = (x[j] - q[j, j + 1:] @ x[j + 1:]) / q[j, j]
    return x


def make(family, n, slices, K=3, S=2, order=4, **kw):
    return PivotProblem(family, n, slices, K, S, order, **kw)


def scaled_denominator(a):
    """(||A||_1, s, Q) with the kernels' scaling rule: s = ceil(log2(||A||_1 / theta13)) squarings, Q = V - U of the
    Pade-13 approximant of A 2^-s."""
    import torch
    from oracle import qoc_oracle as orc
    norm = float(one_norm(a))
    s = max(0, int(math.ceil(math.log2(norm / THETA13)))) if not norm < THETA13 else 0
    at = torch.as_tensor(a * 2.0 ** -s)
    u, v = orc.pade13(at, torch.eye(a.shape[0], dtype=at.dtype))
    return norm, s, (v - u).numpy()


def row_swaps(q):
    """number of row interchanges of LAPACK's partial-pivoting LU (scipy.linalg.lu_factor)."""
    from scipy.linalg import lu_factor
    _, piv = lu_factor(q, check_finite=False)
    return int(np.count_nonzero(piv != np.arange(q.shape[0])))


def factored_matrices(q, own_lu=False):
    """the matrices the kernels factor with partial pivoting for a denominator Q:
      n <= 64           Q itself (row-major LU of tile.cuh);
      n > 64, own LU    the 64 x 64 diagonal blocks of the block LU (k_lg_blockinv), i.e. the leading block and the Schur
                        complements left by the blocks before it - no pivoting between blocks;
      n > 64, cuBLAS    Q^T: getrf reads the row-major Q as column-major."""
    n = q.shape[0]
    if n <= OWN_LU_BLOCK:
        return [q]
    if not own_lu:
        return [q.T]
    out, s = [], np.array(q)
    while s.shape[0] > 0:
        b = min(OWN_LU_BLOCK, s.shape[0])
        out.append(s[:b, :b])
        s = s[b:, b:] - s[b:, :b] @ np.linalg.solve(s[:b, :b], s[:b, b:])
    return out


def slice_report(p, order=None):
    """per slice: (||A||_1, bracket, s, number of row swaps in the matrices the kernels factor).  For n > 64 the plan
    keeps its own block LU only while every slice stays below 2.5 (large.cuh: k_lg_norm_scale raises lu_flag otherwise
    and the plan moves to cuBLAS getrf / getrs for good)."""
    mats = p.magnus_matrices(order)
    reports = [scaled_denominator(a) for a in mats]
    own_lu = p.n > OWN_LU_BLOCK and all(s == 0 and norm < NOPIV_NORM for norm, s, _ in reports) and is_hermitian_problem(p)
    return [(norm, bracket(norm), s, sum(row_swaps(m) for m in factored_matrices(q, own_lu))) for norm, s, q in reports]


def is_hermitian_problem(p):
    return all(is_hermitian(m) for m in p.operators())


# --- the shapes the GPU tests use (tests/test_gpu_pivoting.py); tests/test_pivot_problems_cpu.py checks each of them ------
PER_SLICE_NS = (5, 8, 13, 16, 31, 32, 60, 61, 64)
PER_SLICE = [("H", n, 30, 3, 2, 4) for n in PER_SLICE_NS] + [("N", n, 12, 2, 2, 4) for n in PER_SLICE_NS]

EVAL_CASES = [
    # family, n, slices, K, S, order, F, cost_eval_step, step_target
    ("H", 8, 30, 3, 1, 2, 0, 1, False),
    ("H", 16, 30, 3, 3, 4, 2, 4, True),
    ("H", 32, 30, 3, 5, 6, 0, 1, False),          # S = 5: dense reverse pass
    ("H", 61, 24, 3, 4, 4, 2, 5, True),
    ("H", 64, 24, 3, 8, 4, 0, 1, False),
    ("H", 64, 20, 8, 4, 4, 0, 1, False),          # KR = 8: Magnus M4 with explicit commutator products
    ("H", 64, 20, 3, 1, 6, 3, 3, True),
    ("N", 8, 12, 2, 1, 4, 0, 1, False),
    ("N", 16, 12, 2, 5, 2, 2, 5, True),
    ("N", 32, 16, 2, 3, 6, 0, 1, False),
    ("N", 61, 24, 3, 4, 4, 2, 5, True),
    ("N", 64, 24, 2, 8, 4, 1, 1, False),
    ("N", 64, 16, 8, 4, 4, 0, 1, False),
    ("N", 64, 12, 2, 3, 6, 2, 5, True),
    ("L", 8, 40, 2, 4, 2, 0, 1, False),
    ("L", 16, 40, 2, 1, 4, 2, 3, True),
    ("L", 32, 30, 1, 8, 6, 0, 1, False),
    ("L", 61, 24, 2, 3, 4, 2, 5, True),
    ("L", 64, 24, 4, 4, 4, 0, 1, False),          # KR = 8
    ("L", 64, 20, 2, 5, 6, 2, 3, True),
]

LARGE_CASES = [                                   # H: slices at or above 2.5, so the plan falls back to cuBLAS getrf
    ("H", 65, 12, 3, 2, 4, 2, 5, True),
    ("H", 96, 10, 3, 5, 6, 0, 1, False),
    ("H", 130, 8, 3, 3, 2, 0, 1, False),
    ("H", 256, 8, 3, 2, 4, 0, 1, False),
    ("N", 65, 12, 2, 2, 4, 2, 5, True),
    ("N", 96, 12, 2, 5, 6, 0, 1, False),
    ("N", 130, 12, 2, 3, 2, 0, 1, False),
    ("N", 256, 8, 2, 2, 4, 0, 1, False),
]

# HS at n > 64: the own block LU stays in use; pivots inside its diagonal blocks
LARGE_OWN_LU = [
    ("HS", 65, 16, 3, 2, 4, 2, 5, True),
    ("HS", 96, 12, 3, 5, 6, 0, 1, False),         # dense reverse pass, M6
    ("HS", 130, 12, 3, 3, 2, 0, 1, False),
]

THREE_LEVEL = [("H", 64, 310, 3, 4, 4, 0, 1, False), ("H", 64, 310, 3, 4, 4, 2, 3, True)]
FULL_LENGTH = ("H", 64, 2000, 4, 4, 4, 0, 1, False)
EXPM_NS = (1, 2, 3, 4, 5, 6, 7, 8, 16, 32, 64)
EDGES = (0.5e-13, 2e-13)
EDGE_NS = (16, 64)
# time-sharded (case, world): n <= 64 on both families, n > 64 with the own block LU
TIME_SHARDED = [(("H", 16, 40, 3, 3, 4, 2, 3, True), 3), (("N", 32, 12, 2, 3, 4, 2, 3, True), 2),
                (("HS", 80, 13, 3, 3, 4, 2, 3, True), 2)]
STATE_SHARDED = [("H", 16, 30, 2, 6, 4, 2, 4, True), ("L", 16, 30, 2, 6, 4, 2, 4, True)]
FD_CASES = [("N", 32, 12, 2, 3, 4, 2, 5, True), ("L", 32, 60, 2, 3, 4, 2, 7, True)]
ENSEMBLE = ("H", 16, 24, 3, 2, 4, 0, 1, False)


def expm_stack(n):
    """inputs of the standalone expm / expm_vjp tests: slice matrices of H and N, and (n >= 2) one matrix whose Pade
    denominator needs a row exchange at its first pivot"""
    ps = [PivotProblem("H", n, 30, 3, 1, 4, seed=n)]
    if n > 1:
        ps.append(PivotProblem("N", n, 12, 2, 1, 4, seed=n))
    extra = [vanishing_pivot_matrix(n)[None]] if n > 1 else []
    return np.concatenate([p.magnus_matrices() for p in ps] + extra)


def edge_problem(n, edge):
    return PivotProblem("E", n, 24, 3, 3, 4, F=2, seed=n, cost_eval_step=5, step_target=True, edge=edge)


def from_case(case, seed=None):
    family, n, slices, K, S, order, F, ces, step_target = case
    return PivotProblem(family, n, slices, K, S, order, F=F, seed=n + slices if seed is None else seed, cost_eval_step=ces,
                        step_target=step_target)


def case_id(case):
    family, n, slices, K, S, order, F, ces, step_target = case
    return "%s_n%d_N%d_K%d_S%d_M%d_F%d_ces%d%s" % (family, n, slices, K, S, order, F, ces, "_step" if step_target else "")
