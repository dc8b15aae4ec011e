"""The restatements of tests/digits.py proven against exact arithmetic (Python integers, fractions.Fraction), so that
the GPU tests that hold eg_dev_project_i8 and eg_dev_gemv_i8 to equality with them compare against the right thing."""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

import digits as dg

TOP = Fraction(127, 128)


def _adversarial_columns(n, rng):
    """columns (length n) at the edges of the digit scheme"""
    cols = []
    e = int(rng.integers(-40, 40))
    one_below = np.nextafter(127 / 128, 0)
    for top in (127 / 128, one_below, np.nextafter(127 / 128, 1), 0.5, np.nextafter(0.5, 0), np.nextafter(1.0, 0)):
        c = rng.uniform(-1, 1, n) * top
        c[rng.integers(n)] = top if rng.random() < 0.5 else -top      # the maximum, either sign
        cols.append(np.ldexp(c, e))
    cols.append(np.zeros(n))                                            # zero column
    c = np.zeros(n)
    c[0] = -1.0                                                          # negative maximum alone
    cols.append(c)
    c = np.ldexp(rng.uniform(-1, 1, n), -60)                             # below the last digit of a large entry: rounds to 0
    c[n // 2] = 3.0
    cols.append(c)
    c = rng.uniform(-1, 1, n) * 5e-324 * rng.integers(1, 9, n)           # subnormal entries only
    cols.append(c)
    c = rng.uniform(-1, 1, n)
    c[::3] = rng.uniform(-1, 1, len(c[::3])) * 1e-310                    # mixed normal and subnormal
    cols.append(c)
    cols.append(np.ldexp(rng.uniform(-1, 1, n), int(rng.integers(-500, 500))))
    c = rng.uniform(-1, 1, n)
    c[-1] = 2.0 ** -1021 * 0.75                                          # a column whose maximum is below 2^-1020 ...
    cols.append(c * 2.0 ** -1021 if n > 0 else c)                        # ... scale 0: flushed (documented edge)
    return np.column_stack(cols)


def _cases():
    rng = np.random.default_rng(7)
    out = []
    for n, L in [(1, 1), (2, 3), (7, 5), (31, 40), (33, 17), (64, 9), (70, 40)]:
        U = np.column_stack([_adversarial_columns(n, rng), rng.standard_normal((n, 3)) * 2.0 ** rng.integers(-30, 30, 3)])
        Mt = rng.integers(-1, 2, (L, n)).astype(np.int8)
        Mt[0] = 1                                                        # the largest possible |sum|
        if L > 2:
            Mt[1] = -1
            Mt[2] = 0
        out.append((n, L, U, Mt))
    return out


CASES = _cases()


@pytest.mark.parametrize("case", range(len(CASES)))
def test_colscale_and_digits_against_exact_arithmetic(case):
    n, L, U, Mt = CASES[case]
    e, scale = dg.colscale(U)
    et, st = dg.colscale(torch.from_numpy(U))
    assert np.array_equal(e, et) and np.array_equal(scale, st, equal_nan=True)
    X = dg.integer_digits(U, e)
    assert np.array_equal(X, dg.integer_digits(torch.from_numpy(U), e).numpy())
    for k in range(U.shape[1]):
        m = max(Fraction(abs(float(v))) for v in U[:, k])
        if m == 0:
            assert e[k] == 0 and scale[k] == 0.0
            continue
        r = m / Fraction(2) ** int(e[k])
        # the exponent: [1/2, 127/128), or just below 1/2 after the bump at 127/128
        assert Fraction(1, 2) <= r < TOP or (Fraction(127, 256) <= r < Fraction(1, 2))
        assert scale[k] == math.ldexp(1.0, int(e[k]) - 55)
        if e[k] < -1019:
            assert scale[k] == 0.0                                       # the documented flush
        for i in range(n):
            Xi = int(X[i, k])
            # X reconstructs U to within half a unit of the last digit: 2^(e - 56)
            assert abs(Fraction(Xi) * Fraction(2) ** (int(e[k]) - 55) - Fraction(float(U[i, k]))) <= Fraction(2) ** (int(e[k]) - 56)
            q = dg.balanced_digits(Xi)
            assert sum(d * 256 ** (6 - s) for s, d in enumerate(q)) == Xi
            assert -127 <= q[0] <= 127 and all(-128 <= d <= 127 for d in q[1:])


@pytest.mark.parametrize("case", range(len(CASES)))
def test_restated_product_is_the_correctly_rounded_integer_sum(case):
    n, L, U, Mt = CASES[case]
    e, scale = dg.colscale(U)
    X = dg.integer_digits(U, e)
    B = dg.digits_exact_product(torch.from_numpy(Mt), torch.from_numpy(U), col_block=5).numpy()
    for k in range(U.shape[1]):
        for j in range(L):
            s = sum(int(Mt[j, i]) * int(X[i, k]) for i in range(n))
            if e[k] < -1019:
                ref = 0.0                       # the documented flush: scale 2^(e-55) underflows to 0
            else:
                ref = math.ldexp(float(s), int(e[k]) - 55)   # float(int) rounds correctly; the power-of-two scale is exact
                assert ref == float(s) * scale[k]
            assert B[j, k] == ref, (j, k)
    # the GEMV restatement on single columns: y = (-alpha) (RN(sum m X) 2^(e-55))
    for k in (0, 1, U.shape[1] - 1):
        for alpha in (1.0, -0.3, 0.0):
            y = dg.gemv_exact(torch.from_numpy(Mt), torch.from_numpy(U[:, k].copy()), alpha).numpy()
            assert np.array_equal(y, (-alpha) * B[:, k])


def test_poisoned_column_and_flush():
    U = np.array([[1.0, np.nan, 1e-310, np.inf], [0.5, 2.0, -3e-310, 1.0]])
    e, scale = dg.colscale(U)
    assert e[0] == 1 and scale[0] == 2.0 ** -54 and np.isnan(scale[1]) and np.isnan(scale[3])
    assert e[2] < -1019 and scale[2] == 0.0
    Mt = torch.tensor([[1, -1], [0, 1]], dtype=torch.int8)
    B = dg.digits_exact_product(Mt, torch.from_numpy(U)).numpy()
    assert np.array_equal(B[:, 0], [0.5, 0.5]) and np.isnan(B[:, 1]).all() and np.isnan(B[:, 3]).all()
    assert (B[:, 2] == 0).all()
    # triangular colscale (the scan's U): rows below the diagonal do not count
    T = np.array([[1.0, 0.25], [100.0, 0.5]])
    assert list(dg.colscale(T, full=False)[0]) == [1, 0] and list(dg.colscale(T)[0]) == [7, 0]
