"""GPU parity of the stokes.C shells (C ABI) against the oracle restatement on identical inputs;
bar 1e-12 max-norm relative on random inputs (BASELINE.json north_star).  MatMultPV is also checked componentwise against the
long-double divergence (oracle/highprec.py) with the derived bound C = P_max + 8 + d."""
import numpy as np
import pytest
import torch

import spectral_petsc_b200 as sp
from oracle import highprec as hp
from oracle.stokes import StokesCtx
from conftest import rel_max

pytestmark = pytest.mark.gpu
TOL = 1e-12


def make_pair(dim, cuda, rheology=1, exponent=3.0, eps=1e-2, exact=2, hardness=1.0, gamma0=1.0):
    O = StokesCtx(dim, rheology=rheology, hardness=hardness, exponent=exponent, regularization=eps, gamma0=gamma0, exact=exact)
    U, U2 = O.create_exact_solution()
    G = sp.Stokes(dim, rheology=rheology, hardness=hardness, exponent=exponent, regularization=eps, gamma0=gamma0)
    assert (G.m, G.g, G.gp, G.gv, G.dv) == (O.m, O.g, O.gp, O.gv, O.dv)
    G.set_dirichlet(torch.from_numpy(O.dirichlet.reshape(-1).copy()).to(cuda))
    G.set_force(torch.from_numpy(O.force).to(cuda))
    return O, G, U, U2


CASES = [([8, 6], 0), ([8, 6], 1), ([9, 7, 6], 1), ([16, 16, 16], 0), ([20, 20, 20], 0), ([20, 20, 20], 1), ([33, 10, 12], 1), ([32, 32, 32], 1)]
CASES += [
    ([170, 10], 1),      # an extent past the even-odd reach: deriv_v / deriv_p with DERIV_SUB / DERIV_ADD on AoS strides through the
    ([10, 170], 0),      # dense kernel, crop_nodes_kernel (stokes.cu non-fusable branches), on axis 0 and on the last axis
    ([163, 9, 8], 1),    # the same in 3-D
    ([64, 64, 64], 1),   # m == 2^18 exactly: the largest grid with the fused pad and crop
    ([64, 64, 65], 1),   # above 2^18 with unequal extents: run_jobs split per axis, then crop_sum
    ([63, 64, 65], 0),   # below 2^18 with unequal extents, odd / EXACT / MT-step extents
]


@pytest.mark.parametrize("dim,rheology", CASES, ids=lambda v: str(v))
def test_shells_match_oracle(cuda, dim, rheology):
    O, G, U, U2 = make_pair(dim, cuda, rheology=rheology)
    rng = np.random.default_rng(1)
    xs = 0.3 * rng.standard_normal(O.g)
    Fo = O.function(xs)
    Fg = G.function(torch.from_numpy(xs).to(cuda))
    assert rel_max(Fg.cpu().numpy(), Fo) < TOL
    mn, mx = G.eta_minmax()
    assert mn == pytest.approx(O.min_eta, rel=1e-13) and mx == pytest.approx(O.max_eta, rel=1e-13)
    assert rel_max(G.get_state(0).cpu().numpy(), O.eta) < 1e-13
    if rheology:
        assert rel_max(G.get_state(1).cpu().numpy(), O.deta) < 1e-13
    for j in range(O.d):
        assert rel_max(G.get_state(2 + j).cpu().numpy(), O.strain[j].reshape(-1)) < TOL
    rng = np.random.default_rng(0)
    x = rng.standard_normal(O.g)
    v, p = O.split(x)
    xd = torch.from_numpy(x).to(cuda)
    assert rel_max(G.mat_mult(xd).cpu().numpy(), O.mat_mult(x)) < TOL
    assert rel_max(G.mat_mult_vv(torch.from_numpy(v).to(cuda)).cpu().numpy(), O.mat_mult_vv(v)) < TOL
    pv = G.mat_mult_pv(torch.from_numpy(v).to(cuda)).cpu().numpy()
    assert rel_max(pv, O.mat_mult_pv(v)) < TOL
    ref, M = hp.stokes_divergence(dim, v)
    C = max(dim) + 8 + len(dim)
    r, k = hp.check(pv, ref, M, C)
    print("err/(uM) Stokes PV %s: %.3f" % (dim, r * C))
    assert r <= 1, (r, k)
    assert rel_max(G.mat_mult_vp(torch.from_numpy(p).to(cuda)).cpu().numpy(), O.mat_mult_vp(p)) < TOL
    diag = G.get_diagonal_schur().cpu().numpy()
    eta_in = G.get_state(0).cpu().numpy()[O.int_nodes]
    assert np.all(np.abs(diag - 1.0 / eta_in) <= 2.0 ** -52 * np.abs(1.0 / eta_in))  # 1 / eta of the device's own eta
    if max(dim) <= 160:
        # past 160 points the FFT oracle's strain is off by about 5e-14 relative (its own rounding), which 1 / eta at eta ~ 2e-3
        # carries over the 1e-13 bar; the exact relation above and the eta bar (1e-13) hold there
        assert rel_max(diag, O.get_diagonal_schur()) < 1e-13
    assert np.array_equal(G.mat_mult_host(x), G.mat_mult(xd).cpu().numpy())


def test_K6_null_space_and_exact_residual(cuda):
    # stokes.C:206-212 MatNullSpaceTest: A [0; 1_p] = 0 ; stokes.C:190-196 residual at the exact solution
    O, G, U, U2 = make_pair([20, 20, 20], cuda, rheology=0)
    r = G.function(torch.from_numpy(U).to(cuda)).cpu().numpy()
    assert np.abs(r).max() < 2e-11
    ns = torch.from_numpy(O.merge(np.zeros(O.gv), np.ones(O.gp))).to(cuda)
    assert G.mat_mult(ns).abs().max().item() < 1e-12


def test_pressure_reduce_order_matches_neville(cuda):
    O, G, U, U2 = make_pair([12, 11, 10], cuda)
    rng = np.random.default_rng(3)
    pL = np.zeros(O.m)
    pL[O.int_nodes] = rng.standard_normal(O.gp)
    ref = O.pressure_reduce_order(pL.copy())
    out = G.pressure_reduce_order(torch.from_numpy(pL).to(cuda)).cpu().numpy()
    assert rel_max(out, ref) < TOL


def test_schur_shell_with_callback(cuda):
    O, G, U, U2 = make_pair([9, 8, 7], cuda, rheology=0)
    rng = np.random.default_rng(2)
    p = rng.standard_normal(O.gp)
    # stand-in inner solve: a fixed diagonal scaling (the real one is KSPSolve on MatVV / MatVVPC)
    scale = 1.0 + rng.random(O.gv)
    sd = torch.from_numpy(scale).to(cuda)
    yo = O.mat_mult_schur(p, lambda rhs: rhs * scale)
    yg = G.mat_mult_schur(torch.from_numpy(p).to(cuda), lambda rhs: rhs * sd)
    assert rel_max(yg.cpu().numpy(), yo) < TOL


def test_continuation_rheology_updates(cuda):
    # stokes.C:217-221: the continuation loop changes exponent / regularisation between solves
    from oracle.stokes import continuation_params
    O, G, U, U2 = make_pair([10, 10, 10], cuda, rheology=1, exponent=3.0, eps=1e-4)
    xs = 0.3 * np.random.default_rng(5).standard_normal(O.g)
    for i in range(0, 5):
        e, r = continuation_params(i, 4, 3.0, 1e-4)
        O.set_rheology(e, r)
        G.set_rheology(1, 1.0, e, r, 1.0)
        Fo = O.function(xs)
        Fg = G.function(torch.from_numpy(xs).to(cuda)).cpu().numpy()
        assert rel_max(Fg, Fo) < TOL


def test_errors(cuda):
    with pytest.raises(sp.SB200Error) as ei:
        sp.Stokes([6, 6, 6, 6])
    assert ei.value.code == 56  # stokes.C:1036 "Not implemented for dimension"
    G = sp.Stokes([6, 6])
    with pytest.raises(sp.SB200Error):
        G.set_rheology(2)


@pytest.mark.parametrize("rheology", [0, 1])
def test_full_size_128(cuda, rheology):
    """BASELINE config 5's grid (stokes -rheology 1 -exponent 3 -eps 1e-4 at -dim 128,128,128): StokesFunction (with its cached
    eta / deta / strain) and StokesMatMult against the oracle at the full size - the eo_deriv_kernel<128,...> instantiations on the
    AoS velocity layout inside the Stokes composition."""
    dim = [128, 128, 128]
    O, G, U, U2 = make_pair(dim, cuda, rheology=rheology, exponent=3.0, eps=1e-4)
    xs = 0.3 * np.random.default_rng(1).standard_normal(O.g)
    Fo = O.function(xs)
    Fg = G.function(torch.from_numpy(xs).to(cuda))
    assert rel_max(Fg.cpu().numpy(), Fo) < TOL
    assert rel_max(G.get_state(0).cpu().numpy(), O.eta) < 1e-12
    for j in range(O.d):
        assert rel_max(G.get_state(2 + j).cpu().numpy(), O.strain[j].reshape(-1)) < TOL
    x = np.random.default_rng(0).standard_normal(O.g)
    yo = O.mat_mult(x)
    xd = torch.from_numpy(x).to(cuda)
    y0 = G.mat_mult(xd).clone()
    assert rel_max(y0.cpu().numpy(), yo) < TOL
    # the two evaluation switches at the full size (both on by default; same operator: tests/test_zz4_gpu_optins.py has the small grids)
    for trace, fold in ((True, False), (False, True), (False, False)):
        G.set_trace_divergence(trace)
        G.set_fold_pressure(fold)
        assert rel_max(G.mat_mult(xd).cpu().numpy(), yo) < TOL
        assert rel_max(G.function(torch.from_numpy(xs).to(cuda)).cpu().numpy(), Fo) < TOL
    G.set_trace_divergence(True)
    G.set_fold_pressure(True)
    assert torch.equal(G.mat_mult(xd), y0)
    G.destroy()
