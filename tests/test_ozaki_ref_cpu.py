"""CPU checks of the exact host reference of the INT8 (Ozaki) contraction (tests/ozaki_ref.py) that the bit-exact GPU tests compare
against: the digits represent the fixed-point operands exactly, the segmentation matches the kernels' table, and the folded result
lies within the scheme's error bound of the exact rational product."""
from fractions import Fraction

import numpy as np
import pytest

import ozaki_ref as R


def test_geometry_table():
    """ozaki_geom's segmentation: one segment while S * K fits 65536, otherwise equal segments rounded up to 128 columns."""
    table = {(1, 8): (1, 128, 128), (128, 8): (1, 128, 128), (129, 8): (1, 256, 256), (8192, 8): (1, 8192, 8192),
             (8193, 8): (2, 4224, 4224), (16384, 8): (2, 8192, 8192), (16385, 8): (3, 5504, 5504), (9344, 7): (1, 9344, 9344),
             (9345, 7): (2, 4736, 4736), (8320, 8): (2, 4224, 4224), (65536, 2): (2, 32768, 32768), (300, 2): (1, 384, 384)}
    for (K, S), want in table.items():
        assert R.geometry(K, S) == want, (K, S)
        nseg, Ks, Ksp = want
        assert S * Ks <= 65536 and nseg * Ks >= K and (nseg - 1) * Ks < K


@pytest.mark.parametrize("S", range(2, 9))
def test_digits_represent_the_fixed_point_integer(S):
    """sum_t d_t 256^t == F = rint(a 2^(8S - e)) exactly, every digit in [-128, 127], the most significant one in [-65, 65] (|a| 2^-e
    < 1/4 leaves room for the carries from below), and the planes hold these digits in the kernels' order."""
    rs = np.random.RandomState(S)
    K = 300
    a = R.edge_rows(K, S, rs)
    e = R.row_exponents(a)
    F = R.fixed_point(a, S, e)
    d = R.digits(F, S).astype(np.int64)
    assert (d >= -128).all() and (d <= 127).all()
    assert (np.abs(d[..., S - 1]) <= 65).all()
    back = sum(d[..., t].astype(object) * 256 ** t for t in range(S))
    assert (back == F.astype(object)).all()
    for i in range(a.shape[0]):  # F against exact rational rounding (half to even) of a 2^(8S - e)
        for k in rs.choice(K, 12, replace=False):
            x = Fraction(float(a[i, k])) * Fraction(2) ** (8 * S - int(e[i]))
            assert int(F[i, k]) == round(x), (i, k)
    mx = np.abs(a).max(1)
    nz = mx > 0
    scaled = np.ldexp(mx[nz], -e[nz])
    assert (scaled < 0.25).all() and (scaled >= 0.0625).all()
    ties = np.ldexp(a[5], 8 * S - int(e[5]))  # the tie row: every entry but the maximum is exactly halfway between integers
    assert e[5] == 3 and (np.sum(ties % 1.0 == 0.5) >= K - 1)
    planes, e2 = R.slice(a, S, 0)
    rplanes, _ = R.slice(a, S, 1)
    nseg, Ks, Ksp = R.geometry(K, S)
    assert planes.shape == (a.shape[0], nseg, S, Ksp) and (e2 == e).all()
    assert (planes[:, 0, :, :K] == d[..., ::-1].transpose(0, 2, 1)).all() and not planes[:, 0, :, K:].any()
    assert (rplanes == planes[:, :, ::-1, :]).all()


def test_nonfinite_rows_are_marked():
    """A NaN or an infinity anywhere in a row marks the row (exponent EXP_NONFINITE, zero digits) and NaNs the row / column of V."""
    rs = np.random.RandomState(5)
    a = rs.randn(5, 40)
    a[1, 7], a[3, 0] = np.nan, -np.inf
    b = rs.randn(6, 40)
    b[4, 39] = np.inf
    V, Ap, eA, Bp, eB = R.reference(a, b, 8)
    assert list(eA == R.EXP_NONFINITE) == [False, True, False, True, False] and list(np.nonzero(eB == R.EXP_NONFINITE)[0]) == [4]
    assert not Ap[[1, 3]].any() and not Bp[4].any()
    bad = np.zeros((5, 6), bool)
    bad[[1, 3], :] = True
    bad[:, 4] = True
    assert (np.isnan(V) == bad).all()


@pytest.mark.parametrize("S", range(2, 9))
def test_reference_within_the_scheme_bound_of_the_exact_product(S):
    """|V - a.b| <= 2^(eA+eB) K S (2^-(8S+1) + nseg 2^-56) on sampled entries, against the exact rational product.

    Per term, with a' = a 2^-eA, |a'| < 1/4, rounded to a multiple of 2^-8S (error <= 2^-(8S+1)) and likewise b':
      rounding of the operands   |a~ b~ - a' b'|  <= 2 (1/4) 2^-(8S+1) + 2^-(16S+2)
      dropped products t+u >= S  sum_{w>=S} (2S-1-w) 2^14 256^-(w+2) <= (S-1) 2^-(8S+2) 256/255
    together below S 2^-(8S+1).  The fold adds nseg S correctly rounded terms to partial sums of magnitude < K/15 (the digit expansions
    of a', b' are below 65/256 + 128/256^2 256/255 in magnitude), at most nseg S K 2^-56 in all."""
    rs = np.random.RandomState(100 + S)
    M, N, K = 7, 9, 200
    A = rs.randn(M, K) * np.logspace(-3, 3, M)[:, None]
    B = rs.randn(N, K) * np.logspace(2, -2, N)[:, None]
    B[2] = R.edge_rows(K, S, rs)[5]  # rint ties
    V, Ap, eA, Bp, eB = R.reference(A, B, S)
    nseg = R.geometry(K, S)[0]
    for m in range(M):
        for n in rs.choice(N, 4, replace=False):
            exact = sum(Fraction(float(x)) * Fraction(float(y)) for x, y in zip(A[m], B[n]))
            err = abs(Fraction(float(V[m, n])) - exact) / Fraction(2) ** int(eA[m] + eB[n])
            bound = Fraction(K * S) * (Fraction(1, 2 ** (8 * S + 1)) + Fraction(nseg, 2 ** 56))
            assert err <= bound, (m, n, float(err), float(bound))
    # the truncation is real at small S: the result is not simply the fp64 product
    if S <= 4:
        assert np.abs(V - A @ B.T).max() > 0
