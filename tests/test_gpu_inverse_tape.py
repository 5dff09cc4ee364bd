"""GPU parity of the reverse forms that read the inverse of the Pade denominator from the tape.

Pivot-free slices (Hermitian operators, ||A||_1 < 2.5, no squarings) store Q^-1 in the tape's LU slot, the others the
pivoted LU factors; a family-H plan mixes both formats inside a chunk.  The default variants of the other modules reach the
Krylov reverse pass on either tape and the dense pass at S > 4; this module runs the re-associated rank-S pass
(QOCB_LOWRANK=1) and the dense pass at S <= 4 (QOCB_NO_LOWRANK=1) on the stored and on the recomputed tape.
Oracle: oracle/qoc_oracle.py at 1e-10 relative (cost, final states, gradient)."""
import pytest

from tests import pivot_problems as pp
from tests.test_gpu_pivoting import _assert_oracle, _oracle, _run

pytestmark = pytest.mark.gpu

CASE = ("H", 64, 24, 3, 4, 4, 0, 1, False)


@pytest.mark.parametrize("mode", ["tape", "recompute"])
@pytest.mark.parametrize("env", [{"QOCB_LOWRANK": "1"}, {"QOCB_NO_LOWRANK": "1"}], ids=["lowrank", "dense"])
def test_reverse_forms_on_mixed_tape(env, mode, monkeypatch):
    p = pp.from_case(CASE)
    _assert_oracle(_run(p, env, monkeypatch, store_tape=mode == "tape"), _oracle(p, CASE), pp.case_id(CASE) + "_" + mode)
