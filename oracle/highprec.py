"""Long-double reference of the Chebyshev derivative and of the operator shells built from it (test infrastructure, CPU only).

The FFT restatement in oracle/chebyshev.py carries rounding errors of its own (up to about 1500 u of (|D||x|)_i at P = 170), so
a comparison with it can only use a norm-wise bar.  Here the CGL differentiation matrix is evaluated with mpmath at 40 digits,
rounded once to np.longdouble (64-bit significand), and every product is accumulated in long double.  The reference's own error
is then about 2^-11 of the double-precision unit u = 2^-53 per operation, and a double result can be checked ROW BY ROW against
a bound C * u * M_i, where M_i is a magnitude that bounds every term the computation sums (see `check`).

Layouts follow the rest of the oracle: a field on a d-dimensional grid is row-major (last axis fastest); the derivative along
`axis` acts on the lines of the (O, P, R) factorisation of that array.
"""
import functools

import mpmath
import numpy as np

LD = np.longdouble
U = 2.0 ** -53  # unit roundoff of IEEE double
TINY = 2.0 ** -969  # U * TINY is the smallest normal double (see `check`)
assert np.finfo(LD).eps < 2e-19, "oracle.highprec needs an x87 / quad long double; on this platform np.longdouble is a plain double"

DPS = 40


def _dd_mul(ah, al, bh, bl):
    """(ah + al) * (bh + bl) in double-double arithmetic (Dekker's product), relative error about 2^-104."""

    def split(a):
        c = 134217729.0 * a  # 2^27 + 1
        h = c - (c - a)
        return h, a - h

    p = ah * bh
    ahh, ahl = split(ah)
    bhh, bhl = split(bh)
    e = ((ahh * bhh - p) + ahh * bhl + ahl * bhh) + ahl * bhl
    e = e + (ah * bl + al * bh)
    hi = p + e
    return hi, e - (hi - p)


def _to_dd(values):
    """mpmath numbers -> (hi, lo) double arrays with hi + lo equal to the value to about 2^-106 relative."""
    hi = np.array([float(v) for v in values])
    lo = np.array([float(v - mpmath.mpf(h)) for v, h in zip(values, hi)])
    return hi, lo


def _dd_to_ld(hi, lo):
    """Rounds hi + lo (exactly representable in 106 bits) once to long double."""
    return np.asarray(hi).astype(LD) + np.asarray(lo).astype(LD)


@functools.lru_cache(maxsize=None)
def cgl_matrix(P):
    """The P x P Chebyshev-Gauss-Lobatto differentiation matrix (nodes x_i = cos(i pi / n), n = P - 1) in long double.

    Off the diagonal D_ij = (c_i / c_j) (-1)^(i+j) / (x_i - x_j) with c_0 = c_n = 2, else 1, and x_i - x_j written as
    -2 sin((i+j) t) sin((i-j) t), t = pi / (2n), so no cancellation occurs; the closed-form diagonal is D_00 = (2n^2 + 1) / 6 =
    -D_nn and D_ii = -x_i / (2 (1 - x_i^2)).  (The negative-sum diagonal, exact in exact arithmetic, loses about 4e-17 relative at
    P = 160 when summed in long double.)  The sines and the diagonal are evaluated by mpmath at 40 digits; an off-diagonal
    entry is the product of two reciprocal sines, formed in double-double (106 bits) and then rounded once to long double, so every
    entry is within about 2^-64 relative of the exact value.  Cached per P; the returned array must not be modified."""
    P = int(P)
    if P < 2:
        raise ValueError("the CGL matrix needs P >= 2")
    n = P - 1
    with mpmath.workdps(DPS):
        t = mpmath.pi / (2 * n)
        rs = [mpmath.mpf(0)] + [1 / mpmath.sin(k * t) for k in range(1, 2 * n)]  # 1 / sin(k t), k = 1 .. 2n-1 (all > 0)
        # x_i = 0 exactly at the middle node of odd P (2i = n): its diagonal entry is 0, not the 1e-40 that cos(pi/2) evaluates to
        diag = [mpmath.mpf(2 * n * n + 1) / 6] + [mpmath.mpf(0) if 2 * i == n else -mpmath.cos(2 * i * t) / (2 * mpmath.sin(2 * i * t) ** 2)
                                                   for i in range(1, n)]
        diag.append(-(mpmath.mpf(2 * n * n + 1) / 6))
        rh, rl = _to_dd(rs)
        dh, dl = _to_dd(diag)
    i, j = np.meshgrid(np.arange(P), np.arange(P), indexing="ij")
    off = i != j
    ks = np.where(off, i + j, 1)
    kd = np.where(off, np.abs(i - j), 1)
    hi, lo = _dd_mul(rh[ks], rl[ks], rh[kd], rl[kd])
    c = np.where((i == 0) | (i == n), 2.0, 1.0) / np.where((j == 0) | (j == n), 2.0, 1.0)
    # D_ij = (c_i/c_j) (-1)^(i+j) / (-2 sin((i+j)t) sin((i-j)t)): the factors below are exact powers of two and signs
    f = -0.5 * c * np.where((i + j) % 2 == 1, -1.0, 1.0) * np.sign(i - j)
    D = _dd_to_ld(hi * f, lo * f)
    D[np.arange(P), np.arange(P)] = _dd_to_ld(dh, dl)
    D.setflags(write=False)
    return D


@functools.lru_cache(maxsize=None)
def _abs_matrix(P):
    A = np.abs(cgl_matrix(P))
    A.setflags(write=False)
    return A


def _lines(x, dims, axis):
    dims = [int(v) for v in dims]
    O = int(np.prod(dims[:axis], dtype=np.int64))
    R = int(np.prod(dims[axis + 1:], dtype=np.int64))
    return np.asarray(x).reshape(O, dims[axis], R)


def deriv(x, dims, axis):
    """y = D x along `axis` of the row-major grid `dims`, accumulated in long double (flat long-double array)."""
    X = _lines(x, dims, axis).astype(LD)
    return np.matmul(cgl_matrix(X.shape[1]), X).reshape(-1)


def deriv_mag(x, dims, axis):
    """M = |D| (|x| + |J x|) along `axis`, J the reversal of that axis (flat long-double array).

    It bounds the terms summed by both forms of the derivative: the dense product sum_j D_ij x_j, and the even-odd one,
    sum_j a_ij s_j + b_ij d_j with s_j = x_j + x_{n-j}, d_j = x_j - x_{n-j}, a = (D_ij + D_i,n-j)/2, b = (D_ij - D_i,n-j)/2, since
    |a| |s| + |b| |d| <= (|D_ij| + |D_i,n-j|) (|x_j| + |x_{n-j}|) summed over the pairs is M_i."""
    X = np.abs(_lines(x, dims, axis).astype(LD))
    return np.matmul(_abs_matrix(X.shape[1]), X + X[:, ::-1, :]).reshape(-1)


def check(y, ref, M, C):
    """Worst |y - ref| / (C u M) over the elements, and the flat index where it occurs.  A result passes when the value is <= 1.

    Below the normal range of double (2^-1022) rounding errors are absolute rather than relative: gradual underflow adds at most
    2^-1075 per operation (Higham 2.1), and the long-double reference does not underflow where double does.  M is therefore floored
    at TINY = 2^-969, so the bound never falls below C times the smallest normal double - far above what such errors add up to at
    these sizes, and still 2^-53 below any value of normal size.

    The constant for ONE derivative is C = P + 8.  A dot product of n terms computed in floating point, in any order and with
    or without fused multiply-adds, satisfies |fl(sum a_j b_j) - sum a_j b_j| <= g_n sum |a_j b_j|, g_n = n u / (1 - n u)
    (Higham, Accuracy and Stability of Numerical Algorithms, 3.1).  The dense kernel sums n = P products of the rounded matrix
    entries with x; the even-odd kernel sums n = 2 ceil(P/2) <= P + 1 products a s, b d (the zero padding up to HP adds exact
    zeros).  Against the exact D x this adds the error of each matrix entry (at most 1.25 u relative: the host builds the matrix
    in long double and rounds it to double, tests/test_even_odd_cpu.py) and, for the even-odd form, one rounding of each s_j and
    d_j (u relative to |x_j| + |x_{n-j}|).  All of these terms are bounded by M_i (`deriv_mag`), so
        |y_i - (D x)_i| <= (g_{P+1} (1 + 1.25 u) (1 + u) + 2.25 u + 1.25 u^2) M_i <= (P + 3.26) u M_i   for P <= 300.
    The reference itself is off by at most (P + 1) 2^-64 M_i <= 0.15 u M_i (rounding of D to long double and the long-double
    sums).  C = P + 8 covers both with more than 4 u of room; it is a bound, not a fit to observed errors."""
    y = np.asarray(y, dtype=np.float64).reshape(-1).astype(LD)
    ref = np.asarray(ref, dtype=LD).reshape(-1)
    M = np.asarray(M, dtype=LD).reshape(-1)
    r = np.abs(y - ref) / (LD(C) * LD(U) * np.maximum(M, LD(TINY)))
    k = int(np.argmax(r))
    return float(r[k]), k


# ---- the elliptic operator (elliptic.C:297-339 MatMult_Elliptic, :481-533 FormFunction) ------------------------------------------

def interior_mask(dims):
    """True at the interior nodes of the row-major grid (SetupBC, elliptic.C:386-415: boundary iff any index is on an end)."""
    idx = np.indices([int(v) for v in dims]).reshape(len(dims), -1)
    bdy = np.zeros(idx.shape[1], dtype=bool)
    for j, P in enumerate(dims):
        bdy |= (idx[j] == 0) | (idx[j] == int(P) - 1)
    return ~bdy


def elliptic_pad(dims, U, dirichlet=None):
    """The local field w0: U at the interior nodes in walk order, `dirichlet` (or 0) at the boundary nodes (elliptic.C:305-308, 489-492)."""
    inner = interior_mask(dims)
    w0 = np.zeros(inner.size, dtype=LD)
    w0[inner] = np.asarray(U, dtype=np.float64)
    if dirichlet is not None:
        w0[~inner] = np.asarray(dirichlet, dtype=np.float64)
    return w0


def elliptic_gradient(dims, U, dirichlet):
    """FormFunction's gradient (elliptic.C:489-499): the padded field w0 and, per axis k, (D_k w0, |D_k| (|w0| + |J_k w0|)).
    Check each pair with C = P_k + 8."""
    w0 = elliptic_pad(dims, U, dirichlet)
    return w0, [(deriv(w0, dims, k), deriv_mag(w0, dims, k)) for k in range(len(dims))]


def _divergence_chain(dims, w0, flux):
    """out = sum_k -D_k w_k and its magnitude, with w_k = flux(k, g_k) from g_k = D_k w0 and W_k = flux-magnitude from G_k."""
    d = len(dims)
    out = np.zeros(w0.size, dtype=LD)
    mag = np.zeros(w0.size, dtype=LD)
    for k in range(d):
        w, W = flux(k, deriv(w0, dims, k), deriv_mag(w0, dims, k))
        out -= deriv(w, dims, k)
        mag += deriv_mag(W, dims, k)
    return out, mag


def elliptic_matmult(dims, eta, deta, gradu, U):
    """MatMult_Elliptic: V = crop(-sum_k D_k (eta D_k w0 + deta w0 gradu_k)), w0 = U padded with zero Dirichlet rows.

    eta, deta and gradu (local length m) are inputs, so the device's own cached state can be passed and the check does not
    depend on how pow() was rounded.  Returns (V, M) in long double at the interior nodes; M is the same chain on magnitudes,
    M = sum_k |D_k| (W_k + J_k W_k) with W_k = |eta| |D_k| (|w0| + |J_k w0|) + |deta w0 gradu_k|.

    Check with C = 2 P_max + 16 + d.  Write G_k = |D_k| (|w0| + |J_k w0|) and M_k = |D_k| (W_k + J_k W_k), so M = sum M_k.
    By `check`, the computed first derivative g_k is off by at most (P + 3.41) u G_k; multiplied by eta and differentiated again
    that is at most (P + 3.41) u |D_k| (|eta| G_k) <= (P + 3.41) u M_k.  Forming w_k = eta g_k + deta w0 gradu_k rounds at most three
    times (<= 3.01 u W_k, again <= 3.01 u M_k after |D_k|).  The second derivative of the computed w_k adds (P + 3.41) u M_k (to
    first order).  Summing the d terms in the "0 - T_0 - T_1 ..." chain rounds d - 1 times, <= (d - 1 + 0.01) u M.  In all
    (2 P_max + 9.9 + d) u M, so C = 2 P_max + 16 + d holds with room to spare."""
    eta = np.asarray(eta, dtype=np.float64).astype(LD)
    deta = np.asarray(deta, dtype=np.float64).astype(LD)
    gradu = [np.asarray(g, dtype=np.float64).astype(LD) for g in gradu]
    w0 = elliptic_pad(dims, U)

    def flux(k, g, G):
        c = deta * w0 * gradu[k]
        return eta * g + c, np.abs(eta) * G + np.abs(c)

    out, mag = _divergence_chain(dims, w0, flux)
    inner = interior_mask(dims)
    return out[inner], mag[inner]


def elliptic_residual(dims, eta, U, dirichlet, b):
    """FormFunction: F = crop(-sum_k D_k (eta D_k w0)) - b with w0 = U padded with the Dirichlet values and `eta` given (the
    device's cached one).  Returns (F, M) with M = the magnitude chain of `elliptic_matmult` (deta = 0) plus |b|; the final
    subtraction of b is one more rounding of the chain, so C = 2 P_max + 16 + d holds as derived there."""
    eta = np.asarray(eta, dtype=np.float64).astype(LD)
    w0 = elliptic_pad(dims, U, dirichlet)
    out, mag = _divergence_chain(dims, w0, lambda k, g, G: (eta * g, np.abs(eta) * G))
    inner = interior_mask(dims)
    b = np.asarray(b, dtype=np.float64).astype(LD)
    return out[inner] - b, mag[inner] + np.abs(b)


# ---- the Stokes divergence (stokes.C:557-595 StokesMatMultPV) ------------------------------------------------------------------

def stokes_divergence(dims, v):
    """StokesMatMultPV: sum_i D_i v_i on the velocity zero-padded to the local grid (AoS, component fastest), at the interior
    (pressure) nodes.  Returns (p, M) with M = sum_i |D_i| (|v_i| + |J_i v_i|).

    Each derivative is within (P_i + 3.41) u of its own magnitude (`check`) and the d - 1 additions round d - 1 times, so check
    with C = P_max + 8 + d."""
    dims = [int(P) for P in dims]
    d = len(dims)
    inner = interior_mask(dims)
    vl = np.zeros((inner.size, d), dtype=LD)
    vl[inner] = np.asarray(v, dtype=np.float64).reshape(-1, d)
    out = np.zeros(inner.size, dtype=LD)
    mag = np.zeros(inner.size, dtype=LD)
    for i in range(d):
        vi = np.ascontiguousarray(vl[:, i])
        out += deriv(vi, dims, i)
        mag += deriv_mag(vi, dims, i)
    return out[inner], mag[inner]
