"""GPU parity of MatMult_Elliptic / FormFunction (C ABI) against the oracle restatement of
elliptic.C on identical inputs; bar 1e-12 max-norm relative on random inputs.  Componentwise, the gradient, the MatMult and the
residual are also checked against the long-double reference (oracle/highprec.py) with derived bounds."""
import numpy as np
import pytest
import torch

import spectral_petsc_b200 as sp
from oracle import highprec as hp
from oracle.elliptic import MatElliptic
from conftest import rel_max

pytestmark = pytest.mark.gpu
TOL = 1e-12


def make_pair(dim, gamma, exponent, cuda, exact=2, cos_scale=None):
    O = MatElliptic(dim, gamma=gamma, exponent=exponent)
    u, u2 = O.create_exact_solution(exact, cos_scale=cos_scale)
    G = sp.Elliptic(dim, gamma=gamma, exponent=exponent)
    assert (G.m, G.g, G.nd) == (O.m, O.g, O.nd)
    G.set_dirichlet(torch.from_numpy(O.dirichlet).to(cuda))
    G.set_rhs(torch.from_numpy(O.b).to(cuda))
    return O, G, u, u2


CASES = [([8, 6], 0.0, 2.0), ([8, 6], 4.0, 2.0), ([7, 6, 5], 4.0, 2.0), ([16, 16, 16], 0.0, 2.0), ([16, 16, 16], 4.0, 2.0),
         ([20, 20, 20], 4.0, 3.0), ([12] * 5, 0.0, 2.0), ([12] * 5, 4.0, 2.0), ([5, 4, 3, 6], 1.5, 2.0), ([33, 9], 4.0, 2.0),
         ([3, 3, 3], 4.0, 2.0), ([64, 64, 64], 4.0, 2.0)]

# Grids added for a dispatch branch each, with the launches one MatMult makes there (elliptic.cu matmult_generic).  Fused path
# (d <= 6, every extent <= 160): gradient batch with the pad in its loaders, flux, divergence batch with the crop-sum epilogue = 3
# launches when the extents are equal, 2d + 1 when they are not (one even-odd launch per axis, deriv_eo_jobs), one more (the pad)
# above 2^18 nodes.  Unfused path (d > 6 or an extent > 160): pad, d derivatives, flux, d "-=" derivatives, crop = 2d + 3.
BRANCH = {
    (40,): 3,                     # fused, d = 1: one job, nterms = 0, FormFunction's rhs in the epilogue
    (6,) * 6: 3,                  # fused, d = 6 = SB200_EO_MAX_JOBS: the largest batch, 5 terms in the crop-sum epilogue
    (7, 6, 5, 6, 7, 5): 13,       # fused, d = 6, unequal extents: one launch per axis
    (5, 4, 6, 3, 5, 4, 3): 17,    # unfused, d = 7
    (4,) * 9: 21,                 # unfused, d = 9, m = 2^18 exactly
    (3, 4) * 5: 23,               # unfused, d = 10 (the largest rank)
    (170, 12): 7,                 # unfused, axis 0 on the dense kernel (LEFT tiles, partial last tile)
    (12, 170): 7,                 # unfused, axis 1 on the dense kernel (RIGHT tiles)
    (161, 9, 7): 9,               # unfused, the first extent past the even-odd reach
    (63, 64, 65): 7,              # fused, unequal extents just below 2^18 nodes (fused pad), odd / EXACT / MT-step extents
    (64, 64, 65): 8,              # fused, unequal extents above 2^18: pad_kernel, then one launch per axis
    (65, 65, 65): 4,              # fused, equal extents above 2^18: pad + one batch, odd P (scalar loaders, MT = 5 at P = 65)
    (129, 129, 33): 8,            # fused, unequal extents above 2^18, MT = 9 on axes 0 / 1
}
CASES += [(list(dim), 4.0, 2.0) for dim in BRANCH]


def check_matmult(G, dim, U, V):
    """V = MatMult(U) on the device, componentwise against the long-double chain fed with the device's own eta, deta and gradu
    (C = 2 P_max + 16 + d, oracle.highprec.elliptic_matmult).  Returns max |err| / (u M)."""
    state = [G.get_state(k).cpu().numpy() for k in range(2 + len(dim))]
    ref, M = hp.elliptic_matmult(dim, state[0], state[1], state[2:], U)
    C = 2 * max(dim) + 16 + len(dim)
    r, k = hp.check(V, ref, M, C)
    assert r <= 1, (r, k)
    return r * C


@pytest.mark.parametrize("dim,gamma,exponent", CASES, ids=lambda v: str(v))
def test_function_and_matmult_match_oracle(cuda, dim, gamma, exponent):
    O, G, u, u2 = make_pair(dim, gamma, exponent, cuda)
    rng0, rng1 = np.random.default_rng(0), np.random.default_rng(1)
    # state: residual at a random positive-ish field (SURVEY 8d: scaled so pow(u,p) stays tame)
    Us = 0.1 * rng1.standard_normal(O.g)
    Fo = O.form_function(Us)
    Fg = G.form_function(torch.from_numpy(Us).to(cuda))
    assert rel_max(Fg.cpu().numpy(), Fo) < TOL
    assert rel_max(G.get_state(0).cpu().numpy(), O.eta) < 1e-14
    assert rel_max(G.get_state(1).cpu().numpy(), O.deta) < 1e-14 or np.abs(O.deta).max() == 0
    for k in range(O.d):
        assert rel_max(G.get_state(2 + k).cpu().numpy(), O.gradu[k]) < TOL
    # componentwise: the gradient (C = P_k + 8) and the residual from the device's eta (C = 2 P_max + 16 + d)
    w0, grads = hp.elliptic_gradient(dim, Us, O.dirichlet)
    worst = {}
    for k, (g, M) in enumerate(grads):
        r, i = hp.check(G.get_state(2 + k).cpu().numpy(), g, M, dim[k] + 8)
        assert r <= 1, (k, r, i)
        worst["gradient"] = max(worst.get("gradient", 0.0), r * (dim[k] + 8))
    C = 2 * max(dim) + 16 + len(dim)
    Fr, MF = hp.elliptic_residual(dim, G.get_state(0).cpu().numpy(), Us, O.dirichlet, O.b)
    r, i = hp.check(Fg.cpu().numpy(), Fr, MF, C)
    assert r <= 1, (r, i)
    worst["FormFunction"] = r * C
    U = rng0.standard_normal(O.g)
    Vo = O.mat_mult(U)
    Ud = torch.from_numpy(U).to(cuda)
    n0 = sp.launch_count()
    Vg = G.mat_mult(Ud)
    launches = sp.launch_count() - n0
    assert rel_max(Vg.cpu().numpy(), Vo) < TOL
    worst["MatMult"] = check_matmult(G, dim, U, Vg.cpu().numpy())
    print("err/(uM) elliptic %s: %s" % (dim, ", ".join("%s %.3f" % kv for kv in worst.items())))
    assert np.array_equal(G.mat_mult_host(U), Vg.cpu().numpy())
    # the branch the grid was picked for (the CPU test double launches nothing: launch_count stays 0 there)
    if tuple(dim) in BRANCH and launches:
        assert launches == BRANCH[tuple(dim)], (launches, G.kernel_name())
        assert G.kernel_name().startswith("generic path")


def test_K3_exact2_residual(cuda):
    for dim in ([16, 16, 16], [12] * 5, [20, 20, 20]):
        O, G, u, u2 = make_pair(dim, 0.0, 2.0, cuda)
        r = G.form_function(torch.from_numpy(u).to(cuda)).cpu().numpy()
        assert np.abs(r).max() < 5e-11  # "Norm of exact residual" (elliptic.C:208)


def test_pad_crop_scatter_semantics(cuda):
    # TEST_SCATTER block of elliptic.C:436-456: G->L, D->L, L->G round trips
    O, G, u, u2 = make_pair([6, 5, 4], 0.0, 2.0, cuda)
    U = np.arange(1, O.g + 1, dtype=np.float64)
    L = G.pad(torch.from_numpy(U).to(cuda), with_dirichlet=True).cpu().numpy()
    ref = np.zeros(O.m)
    ref[O.ixG] = U
    ref[O.ixD] = O.dirichlet
    assert np.array_equal(L, ref)
    L0 = G.pad(torch.from_numpy(U).to(cuda), with_dirichlet=False).cpu().numpy()
    ref[O.ixD] = 0.0
    assert np.array_equal(L0, ref)
    assert np.array_equal(G.crop(torch.from_numpy(ref).to(cuda)).cpu().numpy(), U)


def test_full_size_128(cuda):
    dim = [128, 128, 128]
    O, G, u, u2 = make_pair(dim, 4.0, 2.0, cuda)
    assert (G.m, G.g, G.nd) == (2097152, 2000376, 96776)
    Us = 0.1 * np.random.default_rng(1).standard_normal(O.g)
    Fo = O.form_function(Us)
    Fg = G.form_function(torch.from_numpy(Us).to(cuda))
    assert rel_max(Fg.cpu().numpy(), Fo) < TOL
    U = np.random.default_rng(0).standard_normal(O.g)
    Vo = O.mat_mult(U)
    Vg = G.mat_mult(torch.from_numpy(U).to(cuda))
    assert rel_max(Vg.cpu().numpy(), Vo) < TOL
    # linearity at full size
    a = torch.from_numpy(U).to(cuda)
    b = torch.from_numpy(Us).to(cuda)
    lhs = G.mat_mult(3.0 * a - b)
    rhs = 3.0 * G.mat_mult(a) - G.mat_mult(b)
    assert ((lhs - rhs).abs().max() / rhs.abs().max()).item() < 1e-12


@pytest.mark.parametrize("dim", [[32, 32], [32, 32, 32], [64, 64, 64], [32, 32, 32, 32], [128, 128]], ids=lambda v: str(v))
def test_fused_chain_path_matches_generic_and_oracle(cuda, dim):
    # path 1 = generic per-axis kernels, 2 = one chain kernel per axis, 3 = single persistent chain kernel
    O, G, u, u2 = make_pair(dim, 4.0, 2.0, cuda)
    Us = 0.1 * np.random.default_rng(1).standard_normal(O.g)
    O.form_function(Us)
    G.form_function(torch.from_numpy(Us).to(cuda))
    U = np.random.default_rng(0).standard_normal(O.g)
    Vo = O.mat_mult(U)
    Ud = torch.from_numpy(U).to(cuda)
    G.set_path(1)
    V1 = G.mat_mult(Ud).cpu().numpy()
    G.set_path(2)
    V2 = G.mat_mult(Ud).cpu().numpy()
    G.set_path(3)
    V3 = G.mat_mult(Ud).cpu().numpy()
    V3b = G.mat_mult(Ud).cpu().numpy()  # counters re-armed by the previous launch
    assert rel_max(V1, Vo) < TOL
    assert rel_max(V2, Vo) < TOL
    assert rel_max(V3, Vo) < TOL
    assert rel_max(V2, V1) < 1e-13
    assert np.array_equal(V3, V2)  # same arithmetic, same order
    assert np.array_equal(V3, V3b)


@pytest.mark.parametrize("dim", [[96, 96], [96, 96, 96], [48, 48, 48], [80, 80, 80], [112, 112], [112, 112, 112], [144, 144], [160, 160]], ids=str)
def test_persistent_chain_at_96(cuda, dim):
    """Every extent P % 16 == 0 from 32 to 160 runs the persistent chain kernel by default (P = 96: 6 pair tiles; 48 / 80 / 112 / 144: an odd
    number of tiles; 144 / 160: 9 / 10 tiles); against the oracle and the generic path."""
    O, G, u, u2 = make_pair(dim, 4.0, 2.0, cuda)
    Us = 0.1 * np.random.default_rng(1).standard_normal(O.g)
    O.form_function(Us)
    G.form_function(torch.from_numpy(Us).to(cuda))
    U = np.random.default_rng(0).standard_normal(O.g)
    Vo = O.mat_mult(U)
    Ud = torch.from_numpy(U).to(cuda)
    V0 = G.mat_mult(Ud).cpu().numpy()
    assert "persist" in G.kernel_name()
    V0b = G.mat_mult(Ud).cpu().numpy()
    G.set_path(1)
    V1 = G.mat_mult(Ud).cpu().numpy()
    assert rel_max(V0, Vo) < TOL and rel_max(V1, Vo) < TOL and rel_max(V0, V1) < 1e-13
    assert np.array_equal(V0, V0b)
    print("err/(uM) persistent chain %s: %.3f" % (dim, check_matmult(G, dim, U, V0)))


def test_fused_path_rejects_unsupported_extents(cuda):
    G = sp.Elliptic([16, 16, 16])
    G.set_path(2)
    U = torch.zeros(G.g, dtype=torch.float64, device=cuda)
    with pytest.raises(sp.SB200Error) as ei:
        G.mat_mult(U)
    assert ei.value.code == 56
