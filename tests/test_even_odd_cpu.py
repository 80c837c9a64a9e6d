"""The even-odd factorisation the derivative kernels apply (host matrices of sb200_cheb_even_odd, any extent: even, odd, not a multiple
of 16), checked on the CPU with the kernels' own arithmetic: s = u_j + u_{n-j}, d = u_j - u_{n-j}, a = Ae s, b = Bo d,
y_i = a_i + b_i, y_{n-i} = b_i - a_i must equal D u (sb200_cheb_matrix, itself pinned to the reference's ChebMult in tests/test_oracle_ref.py)."""
import numpy as np
import pytest

import spectral_petsc_b200 as sp


@pytest.mark.parametrize("P", [2, 3, 4, 5, 12, 16, 17, 20, 31, 33, 64, 96, 127, 128, 129, 143, 160])
def test_even_odd_halves_reproduce_the_differentiation_matrix(P):
    D = sp.cheb_matrix(P)
    Ae, Bo = sp.cheb_even_odd(P)
    hp, n, hh = Ae.shape[0], P - 1, (P + 1) // 2
    assert hp % 8 == 0 and hp >= hh and hp - hh < 8 and Bo.shape == Ae.shape
    # the padding is zero, and so are the middle node's column of Bo and row of Ae for odd P
    assert not Ae[hh:].any() and not Ae[:, hh:].any() and not Bo[hh:].any() and not Bo[:, hh:].any()
    if P % 2:
        assert not Bo[:, hh - 1].any() and not Ae[hh - 1].any()
    rng = np.random.default_rng(P)
    u = rng.standard_normal((P, 5))
    s, d = np.zeros((hp, 5)), np.zeros((hp, 5))
    for j in range(hh):  # every pair formed the same way, the self-paired middle node of an odd P included
        s[j], d[j] = u[j] + u[n - j], u[j] - u[n - j]
    a, b = Ae @ s, Bo @ d
    y = np.empty_like(u)
    for i in range(hh):
        y[i] = a[i] + b[i]
        y[n - i] = b[i] - a[i] if n - i != i else y[i]
    ref = D @ u
    assert np.abs(y - ref).max() <= 2e-14 * np.abs(ref).max()


def test_kernel_matrix_is_the_rounded_exact_matrix():
    """Every entry of the double matrix the dense kernel applies is within 1.25 u of the exact CGL entry (one rounding to double of a
    long-double value that is itself off by up to about 0.16 u next to the corners, where sinl(pi i / n) is small), which is what the
    bound C = P + 8 of oracle.highprec.check assumes.  An exact zero stays zero: the middle diagonal entry of an odd P (x_i = 0) once
    held about 1e-20, which the dense kernel multiplied into the middle row."""
    from oracle import highprec

    for P in range(2, 301):
        D = sp.cheb_matrix(P)
        ref = highprec.cgl_matrix(P)
        assert np.all(np.abs(D - ref) <= 1.25 * 2.0 ** -53 * np.abs(ref)), P
        if P % 2:
            assert D[P // 2, P // 2] == 0.0


def test_even_odd_matches_the_unpadded_halves_for_multiples_of_16():
    for P in (16, 32, 64, 128):
        D = sp.cheb_matrix(P)
        Ae, Bo = sp.cheb_even_odd(P)
        h = P // 2
        assert Ae.shape == (h, h)
        assert np.abs(Ae - 0.5 * (D[:h, :h] + D[:h, ::-1][:, :h])).max() <= 1e-13 * np.abs(D).max()
        assert np.abs(Bo - 0.5 * (D[:h, :h] - D[:h, ::-1][:, :h])).max() <= 1e-13 * np.abs(D).max()
