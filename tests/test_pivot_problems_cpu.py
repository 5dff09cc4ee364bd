"""CPU preconditions of tests/test_gpu_pivoting.py: the problem families of tests/pivot_problems.py really put slices
into every LU bracket of the kernels, really make partial pivoting swap rows in the matrices the kernels factor (Q for
n <= 64, the diagonal blocks of the own block LU or Q^T for cuBLAS getrf for n > 64), are classified as intended by the
Hermitian rule of qocb_set_operators, and keep the non-unitary evolutions in a range where relative errors mean
something.  Every shape the GPU module uses is checked here; if a builder is simplified so that it stops pivoting,
these tests fail."""
import numpy as np
import pytest
import scipy.linalg as sl

from tests import pivot_problems as pp


def _swap_fraction(rows, lo=pp.SWAP_FROM):
    sel = [r for r in rows if r[0] >= lo]
    return sum(1 for r in sel if r[3] > 0) / max(len(sel), 1)


ALL = (pp.EVAL_CASES + pp.LARGE_CASES + pp.LARGE_OWN_LU + pp.THREE_LEVEL + [pp.FULL_LENGTH] + [c for c, _ in pp.TIME_SHARDED]
       + pp.STATE_SHARDED + pp.FD_CASES + [pp.ENSEMBLE])


def _check_rows(p, rows):
    brackets = {r[1] for r in rows}
    if p.family in ("H", "E"):
        assert brackets == set(pp.BRACKETS), brackets
        assert _swap_fraction(rows) >= 0.25
        # slices the kernels factor WITHOUT pivoting although LAPACK would swap (DESIGN section 3.1)
        assert any(r[1] == "nopiv" and r[3] > 0 for r in rows)
        assert any(r[1] == "scaled" and r[2] >= 1 and r[3] > 0 for r in rows)
    elif p.family == "HS":
        # every slice below 2.5, so that a plan with n > 64 keeps its own block LU; swaps inside its diagonal blocks
        assert brackets == {"lt1.6", "nopiv"}, brackets
        assert _swap_fraction(rows) >= 0.5 and sum(1 for r in rows if r[3] > 0) >= 3
    elif p.family == "N":
        assert {"lt1.6", "pivoted", "scaled"} <= brackets, brackets
        assert _swap_fraction(rows, 0.0) >= 0.25
        assert any(r[1] == "scaled" and r[3] > 0 for r in rows)
    else:
        assert p.family == "L"


@pytest.mark.parametrize("case", ALL, ids=pp.case_id)
def test_brackets_and_swaps(case):
    p = pp.from_case(case)
    _check_rows(p, pp.slice_report(p))


@pytest.mark.parametrize("n", pp.EDGE_NS)
@pytest.mark.parametrize("edge", pp.EDGES)
def test_edge_problems(n, edge):
    p = pp.edge_problem(n, edge)
    _check_rows(p, pp.slice_report(p))
    assert pp.is_hermitian(p.h0) == (edge < 1e-13) and all(pp.is_hermitian(m) for m in p.ops)
    assert not np.array_equal(p.h0, p.h0.conj().T)              # below the rule, but not exactly Hermitian


def test_large_path_factors():
    """what the swap counts above assume about the large path: H problems leave the own-LU regime (plan-wide fallback to
    getrf), HS problems stay in it, and N's Q^T pivots while the transposed shift alone would not"""
    for case in pp.LARGE_CASES + pp.LARGE_OWN_LU:
        p = pp.from_case(case)
        stays = all(s == 0 and norm < pp.NOPIV_NORM for norm, _, s, _ in pp.slice_report(p))
        assert stays == (p.family == "HS"), pp.case_id(case)


@pytest.mark.parametrize("case", pp.PER_SLICE, ids=lambda c: "%s_n%d" % (c[0], c[1]))
def test_per_slice_shapes_pivot(case):
    family, n, slices, K, S, order = case
    rows = pp.slice_report(pp.make(family, n, slices, K=K, S=S, order=order, seed=n))
    assert _swap_fraction(rows, 0.0 if family == "N" else pp.SWAP_FROM) >= 0.25
    assert {"lt1.6", "pivoted", "scaled"} <= {r[1] for r in rows}


@pytest.mark.parametrize("n", pp.EXPM_NS)
def test_standalone_stacks_pivot(n):
    """the standalone expm / expm_vjp inputs: slice matrices of H and N with row swaps (n >= 2)"""
    a = pp.expm_stack(n)
    swaps = sum(1 for m in a if pp.row_swaps(pp.scaled_denominator(m)[2]) > 0)
    assert swaps >= (8 if n > 1 else 0)


@pytest.mark.parametrize("n", [2, 3, 4, 8, 64])
def test_vanishing_pivot_needs_exchange(n):
    """the zero-pivot matrix of the standalone stacks: a solve without row exchange is off by far more than 1e-12,
    the pivoted solve is exact to rounding"""
    import torch
    from oracle import qoc_oracle as orc
    a = pp.vanishing_pivot_matrix(n)
    norm, s, q = pp.scaled_denominator(a)
    assert pp.NOPIV_NORM < norm < pp.THETA13 and s == 0
    assert abs(q[0, 0]) < 1e-8 * abs(q[1, 0]) and pp.row_swaps(q) >= 1
    at = torch.as_tensor(a)
    u, v = orc.pade13(at, torch.eye(n, dtype=at.dtype))
    p_, q_ = (v + u).numpy(), (v - u).numpy()
    want = orc.expm_pade(at).numpy()
    err = lambda x: np.linalg.norm(x - want) / np.linalg.norm(want)
    assert err(sl.solve(q_, p_)) < 1e-14
    assert err(pp.solve_without_exchange(q_, p_)) > 1e-8


def test_classification():
    for case in ALL:
        p = pp.from_case(case)
        assert pp.is_hermitian_problem(p) == (p.family in ("H", "HS")), pp.case_id(case)


def test_is_hermitian_mirror_threshold():
    h = np.array([[1.0, 0.5], [0.5, -1.0]], dtype=complex)
    for rel, want in ((0.9e-13, True), (1.1e-13, False)):
        g = h.copy()
        g[1, 0] += rel * 1.0                       # deviation |a - b| of the pair = rel * max entry (1.0)
        assert pp.is_hermitian(g) == want, rel


def _trajectory_norms(p):
    psi = p.initial_states[..., 0].T
    out = [np.linalg.norm(psi, axis=0)]
    for a in p.magnus_matrices():
        psi = sl.expm(a) @ psi
        out.append(np.linalg.norm(psi, axis=0))
    return np.array(out)


@pytest.mark.parametrize("case", [c for c in ALL if c[0] == "N"], ids=pp.case_id)
def test_nonhermitian_norm_bound(case):
    nr = _trajectory_norms(pp.from_case(case))
    assert nr.min() >= 1e-2 and nr.max() <= 1e2, (nr.min(), nr.max())


def test_loss_family_norms_decay():
    p = pp.make("L", 16, 400, K=2, S=3, order=2, seed=5)
    nr = _trajectory_norms(p)
    assert np.all(np.diff(nr, axis=0) < -1e-6) and nr[-1].min() > np.exp(-1.6)
