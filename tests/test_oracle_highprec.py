"""The long-double reference (oracle/highprec.py) on its own, CPU only: the matrix against an independent mpmath evaluation, exactness
on polynomials, agreement with the FFT restatement, and mutations that the row-wise bound must reject while the 1e-12 max-norm bar
lets some of them through."""
import mpmath
import numpy as np
import pytest

from oracle import highprec as hp
from oracle.chebyshev import ChebCtx, cheb_mult
from conftest import rel_max


def mp_row(P, i, dps=50):
    """Row i of the CGL matrix from the textbook formula (cosine differences, same-row diagonal formula) at `dps` digits."""
    n = P - 1
    with mpmath.workdps(dps):
        x = [mpmath.cos(mpmath.pi * k / n) for k in range(P)]
        c = [2 if k in (0, n) else 1 for k in range(P)]
        row = []
        for j in range(P):
            if j != i:
                row.append(mpmath.mpf(c[i]) / c[j] * (-1) ** (i + j) / (x[i] - x[j]))
            elif i in (0, n):
                row.append((1 if i == 0 else -1) * mpmath.mpf(2 * n * n + 1) / 6)
            else:
                row.append(-x[i] / (2 * (1 - x[i] ** 2)))
        return row


def test_long_double_matrix_matches_mpmath():
    # every P in 2..300; the rows where the formula changes (corners, first / last interior, middle) in full, and the diagonal
    worst = 0.0
    for P in range(2, 301):
        D = hp.cgl_matrix(P)
        n = P - 1
        rows = sorted({0, 1, n // 2, (n + 1) // 2, n - 1, n})
        with mpmath.workdps(50):
            for i in rows:
                ref = mp_row(P, i)
                for j in range(P):
                    e = abs(mpmath.mpf(float(D[i, j])) + mpmath.mpf(float(D[i, j] - hp.LD(float(D[i, j])))) - ref[j])
                    worst = max(worst, float(e / max(abs(ref[j]), mpmath.mpf(1e-30))))  # the middle diagonal entry of odd P is 0
            for i in range(1, n):
                xi = mpmath.cos(mpmath.pi * i / n)
                ref = -xi / (2 * (1 - xi ** 2))
                e = abs(mpmath.mpf(float(D[i, i])) + mpmath.mpf(float(D[i, i] - hp.LD(float(D[i, i])))) - ref)
                worst = max(worst, float(e / max(abs(ref), mpmath.mpf(1e-30))))
    assert worst < 1e-18, worst


@pytest.mark.parametrize("P", [2, 3, 4, 5, 16, 17, 33, 64, 129, 160, 161, 193, 300])
def test_matrix_exact_on_chebyshev_polynomials(P):
    # T_k(cos t) = cos(k t), T_k'(cos t) = k sin(k t) / sin t (k^2 and (-1)^(k+1) k^2 at the ends), k = 0 .. P-1
    n = P - 1
    with mpmath.workdps(40):
        t = [mpmath.pi * m / n for m in range(2 * n)]
        cs = [mpmath.cos(a) for a in t]
        sn = [mpmath.sin(a) for a in t]
        T, dT = [], []
        for i in range(P):
            T.append([cs[(k * i) % (2 * n)] for k in range(P)])
            if i == 0:
                dT.append([mpmath.mpf(k * k) for k in range(P)])
            elif i == n:
                dT.append([mpmath.mpf((-1) ** (k + 1) * k * k) for k in range(P)])
            else:
                dT.append([k * sn[(k * i) % (2 * n)] / sn[i] for k in range(P)])
        Th, Tl = hp._to_dd([v for r in T for v in r])
        dh, dl = hp._to_dd([v for r in dT for v in r])
    T = hp._dd_to_ld(Th, Tl).reshape(P, P)
    dT = hp._dd_to_ld(dh, dl).reshape(P, P)
    D = hp.cgl_matrix(P)
    err = np.abs(D @ T - dT).max(axis=0)
    scale = (np.abs(D) @ np.abs(T)).max(axis=0)
    assert float((err / scale).max()) < 1e-17


@pytest.mark.parametrize("dims,axis", [([2], 0), ([17], 0), ([160, 5], 0), ([4, 170, 3], 1), ([300], 0)], ids=str)
def test_reference_agrees_with_fft_oracle(dims, axis):
    x = np.random.default_rng(7).standard_normal(int(np.prod(dims)))
    ref = hp.deriv(x, dims, axis)
    assert rel_max(cheb_mult(ChebCtx(len(dims), axis, dims), x), ref.astype(np.float64)) < 1e-12


def test_dense_double_product_within_bound():
    # the CPU test double's arithmetic (dense products in double with the same rounded D) sits well inside C = P + 8
    for P in (2, 3, 17, 64, 161, 300):
        x = np.random.default_rng(P).standard_normal(P * 9)
        y = (hp.cgl_matrix(P).astype(np.float64) @ x.reshape(P, 9)).reshape(-1)
        r, _ = hp.check(y, hp.deriv(x, [P, 9], 0), hp.deriv_mag(x, [P, 9], 0), P + 8)
        assert r < 0.5, (P, r)


@pytest.mark.parametrize("P", [17, 33, 65, 129, 161])
def test_check_rejects_mutations(P):
    rng = np.random.default_rng(P)
    R = 9
    x = rng.standard_normal(P * R)
    ref = hp.deriv(x, [P, R], 0)
    M = hp.deriv_mag(x, [P, R], 0)
    C = P + 8
    D = hp.cgl_matrix(P).astype(np.float64)
    good = (D @ x.reshape(P, R)).reshape(-1)
    assert hp.check(good, ref, M, C)[0] < 1
    # 1. one interior element moved by 4 C u M_i: the 1e-12 max-norm bar does not notice, the row-wise bound does
    i = (P // 2 - 1) * R + 3
    bad = good.copy()
    bad[i] += 4 * C * hp.U * float(M[i])
    assert rel_max(bad, ref.astype(np.float64)) < 1e-12
    r, k = hp.check(bad, ref, M, C)
    assert r > 3 and k == i
    # 2. one interior entry of D rounded to float32
    Df = D.copy()
    j = next(j for j in range(1, P) if j != P // 3 and np.float32(D[P // 3, j]) != D[P // 3, j])
    Df[P // 3, j] = np.float32(D[P // 3, j])
    r, k = hp.check((Df @ x.reshape(P, R)).reshape(-1), ref, M, C)
    assert r > 1 and k // R == P // 3
    # 3. odd P: the middle column dropped (the self-paired node of the even-odd form)
    Dm = D.copy()
    Dm[:, (P - 1) // 2] = 0.0
    assert hp.check((Dm @ x.reshape(P, R)).reshape(-1), ref, M, C)[0] > 1


def test_check_below_the_normal_range():
    z = np.zeros(3, dtype=hp.LD)
    assert hp.check(np.zeros(3), z, z, 10) == (0.0, 0)
    # a zero magnitude still rejects anything of normal size, and accepts underflow-sized errors of a few ulps of 2^-1022
    assert hp.check(np.array([0.0, 1e-300, 0.0]), z, z, 10) == (pytest.approx(1e-300 / (10 * 2.0 ** -1022)), 1)
    assert hp.check(np.array([0.0, 3 * 2.0 ** -1074, 0.0]), z, z, 10)[0] < 1e-15


def test_elliptic_and_stokes_references_match_the_oracle():
    from oracle.elliptic import MatElliptic
    from oracle.stokes import StokesCtx

    dims = [9, 7, 6]
    O = MatElliptic(dims, gamma=4.0, exponent=2.0)
    O.create_exact_solution(2)
    rng = np.random.default_rng(3)
    Us = 0.1 * rng.standard_normal(O.g)
    F = O.form_function(Us)
    w0, grads = hp.elliptic_gradient(dims, Us, O.dirichlet)
    for k, (g, Mg) in enumerate(grads):
        assert rel_max(O.gradu[k], g.astype(np.float64)) < 1e-12
    Fr, MF = hp.elliptic_residual(dims, O.eta, Us, O.dirichlet, O.b)
    assert rel_max(F, Fr.astype(np.float64)) < 1e-12
    U = rng.standard_normal(O.g)
    V, MV = hp.elliptic_matmult(dims, O.eta, O.deta, O.gradu, U)
    assert rel_max(O.mat_mult(U), V.astype(np.float64)) < 1e-12
    assert np.all(MV >= np.abs(V)) and np.all(MF >= np.abs(Fr))
    S = StokesCtx([9, 7, 6], rheology=1, exponent=3.0, regularization=1e-2, exact=2)
    v = rng.standard_normal(S.gv)
    p, Mp = hp.stokes_divergence([9, 7, 6], v)
    assert rel_max(S.mat_mult_pv(v), p.astype(np.float64)) < 1e-12
    assert np.all(Mp >= np.abs(p))
