"""CPU tests of the BK_SPARSE host side: the pattern conversion of Context.sparse_pattern (scipy CSR / CSC, Julia's 1-based
colptr / rowval) and the Brusselator Hopf point (examples/brusselator.jl) through the codim-2 host logic with host sparse solvers,
against its closed form."""
import numpy as np
import pytest
import scipy.sparse as sp

import __graft_entry__ as g
from oracle import krylov
from tests import sparse_problems as S
from tests.test_codim2_curves_cpu import NumpyProblem2


@pytest.fixture(scope="module")
def bk():
    return g.load_package()


def _irregular(n=40, seed=0):
    rng = np.random.default_rng(seed)
    A = sp.random(n, n, density=0.1, format="coo", random_state=rng)
    return A


def test_pattern_args_scipy_csr_csc(bk):
    A = _irregular()
    for fmt, M, code in (("csr", A.tocsr(), bk.BK_SPARSE_CSR), ("csc", A.tocsc(), bk.BK_SPARSE_CSC)):
        f, base, nnz, ptr, idx = bk.sparse_pattern_args(M)
        assert (f, base, nnz) == (code, 0, M.nnz)
        assert ptr.dtype == np.int64 and idx.dtype == np.int64 and ptr.flags["C_CONTIGUOUS"] and idx.flags["C_CONTIGUOUS"]
        assert np.array_equal(ptr, M.indptr) and np.array_equal(idx, M.indices)


def test_pattern_args_julia_one_based(bk):
    """SparseMatrixCSC fields passed as they are: ("csc", 1, colptr, rowval)"""
    M = _irregular(seed=1).tocsc()
    colptr, rowval = M.indptr.astype(np.int32) + 1, M.indices.astype(np.int32) + 1
    f, base, nnz, ptr, idx = bk.sparse_pattern_args(("csc", 1, colptr, rowval))
    assert (f, base, nnz) == (bk.BK_SPARSE_CSC, 1, M.nnz)
    assert np.array_equal(ptr, M.indptr + 1) and np.array_equal(idx, M.indices + 1) and ptr.dtype == np.int64
    f2, *_ = bk.sparse_pattern_args((bk.BK_SPARSE_CSR, 0, M.indptr, M.indices))
    assert f2 == bk.BK_SPARSE_CSR


def test_pattern_args_rejects_other_layouts(bk):
    with pytest.raises(bk.BK200Error):
        bk.sparse_pattern_args(_irregular())          # COO
    with pytest.raises(bk.BK200Error):
        bk.sparse_pattern_args(("csc", 2, [0], []))   # base


def test_brusselator_problem_matches_the_example():
    """Jbru_sp is the Jacobian of Fbru! (finite differences), the homogeneous state solves F = 0 for every l, and the closed
    form of the first Hopf point is where a complex pair of the dense spectrum crosses the imaginary axis"""
    par = list(S.BRU_PAR)
    x = S.bru_steady(par) + 0.01 * np.random.default_rng(2).standard_normal(2 * S.BRU_N)
    J = S.bru_J(x, par)
    d = np.random.default_rng(3).standard_normal(2 * S.BRU_N)
    eps = 1e-6
    fd = (S.bru_F(x + eps * d, par) - S.bru_F(x - eps * d, par)) / (2 * eps)
    assert np.linalg.norm(J @ d - fd) < 1e-6 * np.linalg.norm(fd)
    for l in (0.3, 0.51, 0.9):
        assert np.linalg.norm(S.bru_F(S.bru_steady(par), par[:4] + [l])) < 1e-9
    lh, om = S.bru_hopf()
    assert abs(lh - S.BRU_LH) < 1e-12 and abs(om - S.BRU_OMEGA) < 1e-12
    for dl, sign in ((-1e-3, -1), (1e-3, 1)):   # the rightmost pair is stable below l_H, unstable above
        ev, _, _ = S.bru_eigvecs(S.bru_J(S.bru_steady(par), par[:4] + [lh + dl]))
        assert np.sign(ev.real) == sign and abs(ev.imag - om) < 1e-3


def test_brusselator_hopf_newton_host(bk):
    """codim2.newton_hopf on the Brusselator with host sparse-LU solvers reproduces l_H and omega of the closed form to 1e-8"""
    C2, P = bk.codim2, bk.palc
    par = list(S.BRU_PAR)
    l0 = 1.02 * S.BRU_LH
    x0 = S.bru_steady(par)
    par[S.BRU_LENS_L] = l0
    prob = NumpyProblem2(S.bru_F, S.bru_J, x0, par, S.BRU_LENS_L)
    cprob = S.SparseComplexProblem(S.bru_J, par, S.BRU_LENS_L)
    ev, v, w = S.bru_eigvecs(S.bru_J(x0, par))
    opts = P.NewtonPar(tol=1e-10, max_iterations=15, linsolver=krylov.DefaultLS())
    hp = C2.newton_hopf(prob, cprob, x0, l0, ev.imag, v, w, opts, S.sparse_ls2, S.sparse_cls)
    assert hp.converged, hp.residuals
    assert abs(hp.p - S.BRU_LH) < 1e-8 and abs(hp.omega - S.BRU_OMEGA) < 1e-8, (hp.p - S.BRU_LH, hp.omega - S.BRU_OMEGA)
    assert np.linalg.norm(hp.u - x0) < 1e-8


@pytest.mark.parametrize("lam,seed,m", [(0.01, 5, 30), (0.2, 9, 40)])
def test_hessenberg_qr_on_a_shift_invert_spectrum(bk, lam, seed, m):
    """bk_hessenberg_eig on the Arnoldi matrix of (J - 0.5 I)^-1 for the Mittelmann Jacobian (symmetric, double eigenvalues,
    eigenvalues over three decades): the QR iteration with the local deflation test alone stalls on these two (a subdiagonal
    entry just above it; a 2 x 2 block holding a double eigenvalue); the retry converges to the NumPy eigenvalues"""
    import scipy.sparse.linalg as spl
    J = S.Mittelmann().J(np.zeros(S.MIT_N ** 2), [lam])
    lu = spl.splu((J - 0.5 * sp.identity(J.shape[0])).tocsc())
    n = J.shape[0]
    V, H = np.zeros((m + 1, n)), np.zeros((m + 1, m))
    v = np.random.default_rng(seed).standard_normal(n)
    V[0] = v / np.linalg.norm(v)
    for k in range(m):
        w = lu.solve(V[k])
        for _ in range(2):
            h = V[: k + 1] @ w
            w -= V[: k + 1].T @ h
            H[: k + 1, k] += h
        H[k + 1, k] = np.linalg.norm(w)
        V[k + 1] = w / H[k + 1, k]
    ev, _ = bk.hessenberg_eig(H[:m, :m], vectors=False)
    ref = np.linalg.eigvals(H[:m, :m])
    # a double eigenvalue of a nearly defective 2 x 2 block is determined to about sqrt(eps) only
    assert max(np.min(np.abs(ref - e)) for e in ev) < 1e-7 * np.max(np.abs(ref))
