"""CPU checks of the equilibration reference (tests/equilibrate_ref.py) against LAPACK: the power-of-two scales equal
scipy's dgeequb bit for bit, dlaqge's EQUED decision, and the emulated refinement it is for."""
import math

import numpy as np
import pytest
from scipy.linalg import lapack

import equilibrate_ref as eq


def spread_matrix(rng, n, spread):
    return (rng.standard_normal((n, n)) * (2.0 ** rng.uniform(-spread, spread, n))[:, None]
            * (2.0 ** rng.uniform(-spread, spread, n))[None, :])


def assert_matches_lapack(A):
    r, c, rowcnd, colcnd, amax, info = eq.geequb_pow2(A)
    R, Cs, rc, cc, am, inf = lapack.dgeequb(A)
    assert info == inf
    assert np.array_equal(r, R) and np.array_equal(c, Cs)
    assert (rowcnd, colcnd, amax) == (rc, cc, am)


@pytest.mark.parametrize("spread", [0, 4, 12, 30])
def test_scales_equal_dgeequb_on_random_matrices(spread):
    rng = np.random.default_rng(spread)
    for _ in range(40):
        A = spread_matrix(rng, int(rng.integers(2, 60)), spread)
        assert_matches_lapack(A)


def test_scales_equal_dgeequb_at_exact_powers_of_two():
    for e in range(-60, 61):
        A = np.full((3, 3), 0.25)
        A[1, 2] = 2.0 ** e  # row 1's maximum, and column 2's after the row scaling
        assert_matches_lapack(A)
        assert_matches_lapack(A * 0.75)  # f = 0.75: between two powers


def test_scales_equal_dgeequb_with_rectangular_looking_spreads():
    """rows spread wide, columns not (and the other way round): only one side ends up badly scaled"""
    rng = np.random.default_rng(7)
    n = 48
    rows = 2.0 ** rng.integers(-30, 31, n)
    A = rng.standard_normal((n, n)) * rows[:, None]
    assert_matches_lapack(A)
    assert_matches_lapack(np.ascontiguousarray(A.T))
    assert eq.equilibrate(A)[0] in (1, 3) and eq.equilibrate(A.T)[0] in (2, 3)


def test_zero_row_or_column_means_no_equilibration():
    rng = np.random.default_rng(3)
    A = spread_matrix(rng, 20, 10)
    Z = A.copy()
    Z[5, :] = 0.0
    assert eq.geequb_pow2(Z)[5] == lapack.dgeequb(Z)[5] == 6
    Z2 = A.copy()
    Z2[:, 7] = 0.0
    assert eq.geequb_pow2(Z2)[5] == lapack.dgeequb(Z2)[5] == 20 + 8
    for M in (Z, Z2):
        e, r, c = eq.equilibrate(M)
        assert e == 0 and (r == 1).all() and (c == 1).all()
    N = A.copy()
    N[3, 4] = np.nan
    assert eq.equilibrate(N)[0] == 0
    N[3, 4] = np.inf
    assert eq.equilibrate(N)[0] == 0


@pytest.mark.parametrize("rowcnd,colcnd,amax,expect", [
    (0.1, 0.1, 1.0, "N"), (0.0625, 0.1, 1.0, "R"), (0.1, 0.0625, 1.0, "C"), (0.0625, 0.0625, 1.0, "B"),
    (1.0, 1.0, eq.SMALL, "N"), (1.0, 1.0, eq.SMALL / 2, "R"), (1.0, 1.0, eq.LARGE, "N"), (1.0, 1.0, eq.LARGE * 2, "R"),
    (1.0, 0.09999, eq.LARGE * 2, "B"),
])
def test_laqge_decision(rowcnd, colcnd, amax, expect):
    assert eq.laqge_equed(rowcnd, colcnd, amax) == expect


def test_laqge_decision_on_constructed_matrices():
    one = np.eye(4) + 0.5
    assert eq.equilibrate(one)[0] == 0
    # row maxima 1.5 and 1.5 * 2^-5: rounded to 1 and 2^-4 (int() truncates log2 toward zero), ROWCND 1/16 < 0.1
    rows = one * np.array([1.0, 1.0, 1.0, 2.0 ** -5])[:, None]
    assert eq.equilibrate(rows)[0] in (1, 3)
    near = one * np.array([1.0, 1.0, 1.0, 2.0 ** -4])[:, None]   # ROWCND 1/8 >= 0.1: left alone
    e, _, _ = eq.equilibrate(near)
    assert e & 1 == 0
    cols = one * np.array([1.0, 2.0 ** -6, 1.0, 1.0])[None, :]  # COLCND 1/16 after the row scales (row 1: r = 2)
    assert eq.equilibrate(cols)[0] == 2
    both = rows * np.array([1.0, 2.0 ** -9, 1.0, 1.0])[None, :]
    assert eq.equilibrate(both)[0] == 3


def test_equilibrated_refinement_keeps_fp16_in_range(oracle):
    """the emulation: rows and columns spread by 2^+-10 overflow fp16 unscaled, and converge once equilibrated"""
    rng = np.random.default_rng(0)
    n = 256
    A0 = rng.standard_normal((n, n)) + 2 * math.sqrt(n) * np.eye(n)
    A = (2.0 ** rng.integers(-10, 11, n))[:, None] * A0 * (2.0 ** rng.integers(-10, 11, n))[None, :]
    b = A @ rng.standard_normal(n)
    with np.errstate(all="ignore"):
        plain = oracle.refine(A, b, oracle.lu_mixed_emulated(A, nb=128))
    assert not plain["converged"]
    e, r, c = eq.equilibrate(A)
    assert e == 3
    s = eq.refine_equilibrated(oracle, A, b, r, c)
    base = oracle.refine(A0, A0 @ rng.standard_normal(n), oracle.lu_mixed_emulated(A0, nb=128))
    assert s["converged"] and s["iters"] <= base["iters"] + 1, (s["iters"], base["iters"])
