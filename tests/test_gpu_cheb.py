"""GPU parity of the Chebyshev derivative (C ABI -> DMMA kernels) against the oracle's restated
FFTW path, on random N(0,1) inputs, max-norm relative, bar 1e-12 (BASELINE.json north_star), and row by row against the
long-double reference (oracle/highprec.py) with the derived bound C = P + 8."""
import numpy as np
import pytest
import torch

import spectral_petsc_b200 as sp
from oracle import highprec as hp
from oracle.chebyshev import PI, ChebCtx, cheb_mult
from conftest import rel_max

pytestmark = pytest.mark.gpu
TOL = 1e-12

SHAPES = [
    ([2], 0), ([3], 0), ([5], 0), ([12], 0), ([16], 0), ([33], 0), ([128], 0), ([129], 0), ([200], 0), ([300], 0),
    ([8, 7, 6], 0), ([8, 7, 6], 1), ([8, 7, 6], 2),
    ([6, 5, 7, 3], 0), ([6, 5, 7, 3], 1), ([6, 5, 7, 3], 2),           # AoS velocity layout stokes.C:284-289
    ([20, 20, 20, 3], 0), ([20, 20, 20, 3], 1), ([20, 20, 20, 3], 2),
    ([16, 16, 16], 0), ([16, 16, 16], 1), ([16, 16, 16], 2),
    ([12] * 5, 0), ([12] * 5, 1), ([12] * 5, 2), ([12] * 5, 3), ([12] * 5, 4),
    ([40, 3, 70], 1), ([3, 130, 5], 1), ([1, 64, 1], 1), ([17, 1, 9], 0),
    ([128, 128, 128], 0), ([128, 128, 128], 1), ([128, 128, 128], 2),
    ([64, 64, 64, 3], 0), ([64, 64, 64, 3], 1), ([64, 64, 64, 3], 2),
]


def _edge_shapes():
    """Every tile edge of the derivative kernels.  Even-odd kernel (P <= 160): MT = ceil(ceil(P/2)/8) steps at P = 16k+1 and the
    EXACT instantiation runs at P = 16 MT, so 16k-1 / 16k / 16k+1 for k = 1..10, plus the smallest extents 2, 3, 4.  Dense kernel:
    161 (first extent past the even-odd reach), 162, 192 / 193 (the padded extent Pp grows past 192) and 257.  Layouts per P:
    [P] (one line), [P, 24] on axis 0 (R % 8 == 0: 16-byte block loader), [P, 13] on axis 0 (scalar loader, partial last 8-line
    block), [5, P, 3] on axis 1 (O > 1 with a short R); for P > 160 also [P, 70] on axis 0 (dense LEFT tiles with a partial last tile)
    and [9, P, 5] on axis 1 (dense RIGHT tiles with several o-groups per tile)."""
    Ps = [2, 3, 4] + [16 * k + e for k in range(1, 11) for e in (-1, 0, 1)] + [161, 162, 192, 193, 257]
    out = []
    for P in Ps:
        out += [([P], 0), ([P, 24], 0), ([P, 13], 0), ([5, P, 3], 1)]
        if P > 160:
            out += [([P, 70], 0), ([9, P, 5], 1)]
    return [s for s in out if s not in SHAPES]


SHAPES += _edge_shapes()
EO_MAX_P = 160  # extents the even-odd kernel takes (deriv_eo.cu: HP <= 80); larger ones run the dense deriv_kernel


@pytest.mark.parametrize("dims,tr", SHAPES, ids=lambda v: str(v))
def test_cheb_mult_matches_oracle(cuda, dims, tr):
    rng = np.random.default_rng(abs(hash((tuple(dims), tr))) % (2 ** 31))
    x = rng.standard_normal(int(np.prod(dims)))
    ref = cheb_mult(ChebCtx(len(dims), tr, dims), x)
    A = sp.Cheb(len(dims), tr, dims)
    xd = torch.from_numpy(x).to(cuda)
    y = A.mult(xd)
    torch.cuda.synchronize()
    assert torch.equal(xd.cpu(), torch.from_numpy(x))  # x preserved (chebyshev.c:127)
    assert rel_max(y.cpu().numpy(), ref) < TOL
    # row by row against the long-double reference, C = P + 8 (derivation in oracle.highprec.check)
    P = dims[tr]
    r, k = hp.check(y.cpu().numpy(), hp.deriv(x, dims, tr), hp.deriv_mag(x, dims, tr), P + 8)
    print("err/(uM) %s derivative %s axis %d: %.3f at %d" % ("even-odd" if P <= EO_MAX_P else "dense", dims, tr, r * (P + 8), k))
    assert r <= 1, (r, k)
    # host-buffer entry point (the e2e path) gives the same bits
    assert np.array_equal(A.mult_host(x), y.cpu().numpy())


@pytest.mark.parametrize("dims,tr", [([17, 24], 0), ([32, 8], 0), ([33, 16], 0), ([64, 40], 0), ([129, 24], 0), ([160, 8], 0), ([6, 48, 16], 1),
                                     ([193, 24], 0), ([5, 170, 8], 1)], ids=str)
def test_misaligned_views_give_the_same_bits(cuda, dims, tr):
    """x and y as views one element into larger buffers (8-byte but not 16-byte aligned): a shape with R % 8 == 0 that normally takes
    the even-odd kernel's 16-byte block loader runs its scalar loader instead.  Both fill the same shared-memory layout and the GEMM
    and epilogue arithmetic are the same, so the result must be bit-identical to the aligned call (the dense kernel, P > 160, too)."""
    n = int(np.prod(dims))
    rng = np.random.default_rng(n + tr)
    x = torch.from_numpy(rng.standard_normal(n)).to(cuda)
    A = sp.Cheb(len(dims), tr, dims)
    y = A.mult(x)
    xbuf = torch.zeros(n + 3, dtype=torch.float64, device=cuda)
    ybuf = torch.full((n + 3,), 7.0, dtype=torch.float64, device=cuda)
    xv = xbuf[1:1 + n]
    xv.copy_(x)
    yv = ybuf[1:1 + n]
    assert xv.data_ptr() % 16 == 8 and yv.data_ptr() % 16 == 8
    A.mult(xv, yv)
    torch.cuda.synchronize()
    assert torch.equal(yv, y)
    assert ybuf[0].item() == 7.0 and torch.equal(ybuf[1 + n:], torch.full((2,), 7.0, dtype=torch.float64, device=cuda))


def test_K1_K2_analytic(cuda):
    m1 = 5
    u = np.exp(np.cos(np.arange(m1) * PI / (m1 - 1)))
    y = sp.Cheb(1, 0, [m1]).mult_host(u)
    assert np.abs(y - u).max() == pytest.approx(1.0293308609854e-02, rel=1e-9)
    m, n, p = 8, 7, 6
    x, yy, z = (np.cos(np.arange(k) * PI / (k - 1)) for k in (m, n, p))
    a = np.exp(x)[:, None, None] + np.exp(yy)[None, :, None] + np.exp(z)[None, None, :]
    ex = [np.exp(x)[:, None, None], np.exp(yy)[None, :, None], np.exp(z)[None, None, :]]
    for d, expect in enumerate((6.245e-06, 8.72e-05, 1.04e-03)):
        out = sp.Cheb(3, d, [m, n, p]).mult_host(a.ravel()).reshape(a.shape)
        assert np.abs(out - ex[d]).max() == pytest.approx(expect, rel=5e-3)


def test_linearity_and_constants_full_size(cuda):
    # size-independent properties at BASELINE's full size: D(1) = 0, D(x_axis) = 1, linearity
    P = 128
    for tr in range(3):
        A = sp.Cheb(3, tr, [P, P, P])
        ones = torch.ones(P ** 3, dtype=torch.float64, device=cuda)
        y = A.mult(ones)
        assert y.abs().max().item() < 1e-9  # |D| row sums ~ 1e4, eps-level cancellation
        xs = torch.cos(torch.arange(P, dtype=torch.float64, device=cuda) * PI / (P - 1))
        shape = [1, 1, 1]
        shape[tr] = P
        X = xs.reshape(shape).expand(P, P, P).contiguous().reshape(-1)
        assert (A.mult(X) - 1.0).abs().max().item() < 1e-9
        g = torch.Generator(device="cuda").manual_seed(tr)
        a = torch.randn(P ** 3, dtype=torch.float64, device=cuda, generator=g)
        b = torch.randn(P ** 3, dtype=torch.float64, device=cuda, generator=g)
        lhs = A.mult(2.0 * a + b)
        rhs = 2.0 * A.mult(a) + A.mult(b)
        assert ((lhs - rhs).abs().max() / rhs.abs().max()).item() < 1e-13


def test_errors(cuda):
    with pytest.raises(sp.SB200Error) as ei:
        sp.Cheb(2, 2, [4, 4])
    assert ei.value.code == 83
    A = sp.Cheb(1, 0, [8])
    x = torch.zeros(8, dtype=torch.float64, device=cuda)
    with pytest.raises(sp.SB200Error):
        A.mult(x, x)  # x != y required
