"""The dense-system families of tests/local_solver_cases.py drive the pivoting paths of the blocked solver they are
meant for (checked by the NumPy replay of its panel decisions), and the extended-precision reference solve is
accurate (checked against mpmath at 50 digits).  CPU only: the GPU runs are in test_zz_local_solvers_gpu.py."""
import mpmath
import numpy as np
import pytest

import local_solver_cases as lc

NS = [1, 2, 3, 4, 5, 7, 8, 9, 12, 15, 16, 17, 31, 33, 47, 48, 111, 112]


def _npanel(n):
    return (n + 3) // 4


@pytest.mark.parametrize("n", NS)
def test_family_f_fast_on_every_panel(n):
    for seed in range(3):
        assert lc.panel_paths(lc.family_f(n, seed)) == ["fast"] * _npanel(n)


@pytest.mark.parametrize("n", [n for n in NS if n >= 8])
def test_family_s_slow_on_every_panel(n):
    M = lc.family_s(n)
    assert lc.panel_paths(M) == ["slow"] * _npanel(n)
    # panel 0's natural block is exactly singular
    assert not np.any(M[:4, :4])
    assert lc.cond_inf(M) < 1e3


@pytest.mark.parametrize("n", [n for n in NS if n >= 2])
def test_family_m_only_panel_k_slow(n):
    Q = _npanel(n)
    for k in sorted({0, Q // 2, Q - 1}):
        if n - 4 * k < 2:
            continue
        exp = ["fast"] * Q
        exp[k] = "slow"
        M = lc.family_m_panel(n, k)
        assert lc.panel_paths(M) == exp, k
        assert lc.cond_inf(M) < 1e4


@pytest.mark.parametrize("n", [n for n in NS if n >= 8])
def test_family_m_gaussian_mixes_paths(n):
    paths = set()
    for seed in range(lc.GAUSS_SEEDS):
        paths.update(lc.panel_paths(lc.family_m_gauss(n, seed)))
    assert paths == {"fast", "slow"}


@pytest.mark.parametrize("n", [2, 3, 4, 5, 9, 16, 33, 112])
def test_family_g_growth_on_the_threshold(n):
    for target, path in lc.G_TARGETS:
        M = lc.family_g(n, target)
        g = lc.panel_growth(M)
        assert abs(g - target) <= 1e-9 * target, (target, g)
        assert lc.panel_paths(M)[0] == path, target
    # the float rounding decides the middle pair: above 64 in double, one rounds down to 64 and one does not
    assert np.float32(64.0 + 3e-6) == 64.0 and np.float32(64.0 + 5e-6) > 64.0


@pytest.mark.parametrize("n", NS)
def test_family_c_grades_one_panel(n):
    q = lc.graded_panel(n)
    for e in lc.C_EXPONENTS:
        M, Mu, d = lc.family_c(n, e)
        assert np.allclose(M, Mu * d[None, :], rtol=0, atol=0)
        exp = ["fast"] * _npanel(n)
        if e >= 3 and n > 4:   # for n <= 4 every column is graded and the row scaling undoes it
            exp[q] = "slow"
        assert lc.panel_paths(M) == exp, e
        assert lc.panel_paths(Mu) == ["fast"] * _npanel(n)


@pytest.mark.parametrize("n", [n for n in NS if n >= 2])
def test_singular_families_are_singular(n):
    cases = [lc.singular_duplicate_row(n), lc.singular_zero_column(n)]
    if n % 4 == 3:
        cases.append(lc.singular_last_panel(n))
    for M in cases:
        assert np.linalg.matrix_rank(M) < n
        # every row has unit 1-norm (as the assembly's rows do)
        assert np.allclose(np.abs(M).sum(axis=1), 1.0)
    # the rank deficiency of singular_last_panel lies in its last, partial panel only
    if n % 4 == 3 and n > 3:
        M = lc.singular_last_panel(n)
        assert np.linalg.matrix_rank(M[: n - 3, : n - 3]) == n - 3
    # LAPACK's LU meets an exact zero pivot on each (the reference's np.linalg.inv raises)
    for M in cases:
        with pytest.raises(np.linalg.LinAlgError):
            np.linalg.inv(M)


def test_sizes_cover_every_remainder():
    s = lc.sizes(112)
    assert s[:9] == list(range(1, 10)) and s[-2:] == [111, 112]
    assert {x % 4 for x in s} == {0, 1, 2, 3}
    assert {x % 32 for x in s} >= {31, 0, 1}
    assert lc.sizes(16) == [1, 2, 3, 4, 5, 6, 7, 8, 9, 15, 16]


def _mp_solve(M, B):
    mpmath.mp.dps = 50
    Mm = mpmath.matrix(M.tolist())
    X = np.zeros_like(B)
    for c in range(B.shape[1]):
        x = mpmath.lu_solve(Mm, mpmath.matrix(B[:, c].tolist()))
        X[:, c] = [float(v) for v in x]
    return X


@pytest.mark.parametrize("make", [lambda: lc.family_f(7), lambda: lc.family_m_gauss(9, 1), lambda: lc.family_s(8),
                                  lambda: lc.family_g(6, 64.0 + 5e-6), lambda: lc.family_c(9, 12)[0],
                                  lambda: lc.family_m_panel(12, 1)])
def test_reference_solve_against_mpmath(make):
    M = make()
    B = lc.rhs(M.shape[0], 3)
    X = lc.ref_solve(M, B)
    Xm = _mp_solve(M, B)
    # the refined solution is the correctly rounded one up to a few units in the last place
    assert np.abs(X - Xm).max() <= 4 * lc.U * np.abs(Xm).max()
    # and never further from it than plain float64 LU
    assert np.abs(X - Xm).max() <= np.abs(np.linalg.solve(M, B) - Xm).max()


def test_error_ratio_definition():
    M = lc.family_f(5)
    X = lc.ref_solve(M, lc.rhs(5, 2))
    assert lc.error_ratio(X, X, M) == 0.0
    bound = 50 * 5 * lc.U * lc.cond_inf(M)
    assert lc.error_ratio(X * (1 + 2 * bound), X, M) == pytest.approx(2.0, rel=1e-2)
