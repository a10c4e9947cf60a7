"""The oracle's reduced-camera-system solve (orc_ldlt_solve: the LDL^T without pivoting behind every LocalBA parity test) against a
high-precision referee, and the referee's own generators. CPU only."""
import numpy as np
import pytest

from . import ba_solve_ref as R

SIZES = [1, 6, 31, 32, 33, 64, 294, 383, 546, 774]


@pytest.mark.parametrize("fam", ["dense_spd", "ba_shaped", "graded"])
@pytest.mark.parametrize("n", SIZES)
def test_oracle_ldlt_meets_the_gates(oracle, fam, n):
    S = R.FAMILIES[fam](n); g = R.rhs(n)
    xs = R.reference_solve(S, g)
    x, ok = oracle.ldlt_solve(S, g)
    assert ok
    assert R.backward_error(S, g, x) <= 8 * n * R.U
    assert R.backward_error(S, g, xs) <= R.U                       # the referee itself
    if fam != "graded":
        assert R.forward_error(x, xs) <= R.kappa_inf(S) * n * R.U


def test_oracle_ldlt_reads_the_lower_triangle_only(oracle):
    S = R.ba_shaped(60); g = R.rhs(60)
    P = S.copy(); P[np.triu_indices(60, 1)] = np.nan
    x0, _ = oracle.ldlt_solve(S, g)
    x1, ok = oracle.ldlt_solve(P, g)
    assert ok and np.array_equal(x0.view(np.uint64), x1.view(np.uint64))


@pytest.mark.parametrize("n", [40, 546])
def test_oracle_ldlt_reports_bad_pivots(oracle, n):
    S = R.dense_spd(n); g = R.rhs(n)
    assert oracle.ldlt_solve(S, g)[1]
    for k in (0, 31, 32, 33, n - 1):
        assert not oracle.ldlt_solve(R.zero_pivot(S, k), g)[1], k
    for k in (0, 33, n - 1):
        B = S.copy(); B[k, k] = np.nan
        assert not oracle.ldlt_solve(B, g)[1], k


@pytest.mark.parametrize("n", [12, 60, 294, 546])
def test_generators_hit_their_conditioning(n):
    assert np.linalg.cond(R.dense_spd(n)) < 6                       # eigenvalues of M M^T / n + I lie in [1, ~5]
    for kappa in (1e2, 1e4, 1e6):
        S = R.ba_shaped(n, kappa=kappa)
        assert np.allclose(S, S.T, rtol=0, atol=0)
        assert 0.9 * kappa < np.linalg.cond(S) < 1.1 * kappa, kappa
    G = R.graded(n)
    d = np.diag(G) / np.diag(R.dense_spd(n))
    assert d.min() < 1e-2 and d.max() > 1e2 and np.linalg.eigvalsh(G)[0] > 0
